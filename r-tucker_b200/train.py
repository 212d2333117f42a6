"""Epoch driver with the reference's function surface (train.py:37-42, 69-167) over the fused path.

  extract_tensor(model)                                              train.py:37-42
  train_one_epoch(model, optimizer, criterion, train_loader, reg)    train.py:69-91
  evaluate(model, criterion, dataloader)                             train.py:94-125
  train(model, optimizer, train_loader, val_loader, test_loader, config, regulizer, scheduler)   train.py:128-167

Differences that follow from the fused path: the loaders are ``data.DeviceEpoch`` objects (device-resident CSR
epoch, on-device shuffle) yielding ``(features, SparseTargets)``; the loss closure is a ``FusedLoss``; losses and
gradient norms are accumulated in device scalars and read back ONCE per epoch (the reference formats a device
tensor into its tqdm bar every step, train.py:88: an implicit synchronisation per step); checkpoints carry the
optimiser state (checkpoint.py).  ``criterion`` selects the training objective among the two the fused kernels
implement: ``nn.BCELoss(reduction="mean")`` (train.py:136, the default) and ``nn.CrossEntropyLoss(reduction="mean")``
(1-N softmax cross-entropy over all entities; no ``weight``, no ``ignore_index``, ``label_smoothing=0``: the smoothing
comes from the loader, as for the BCE).  Evaluation is the same for both unless asked otherwise: the reference's BCE
evaluation loss and the probability-space filtered ranks.  ``evaluate(space="logit")`` / ``train(eval_space="logit")``
rank the exact logits and report the cross-entropy instead, which is what a cross-entropy model needs: its top logits
sit where the fp32 sigmoid has saturated to 1.0.
"""
import os
import time

import torch
from torch import nn

from . import checkpoint
from .evaluation import _check_space, _sums_from_ranks, rank_batch
from .manifold import SFTucker, Tucker
from .engine import RelationTerm
from .optim import FusedLoss
from .rank import set_rank


def extract_tensor(model):
    """train.py:37-42 -- factor order (relation, subject, object); SF-Tucker shares the last two."""
    if model.symmetric:
        return SFTucker(model.core.data, [model.R.weight], num_shared_factors=2, shared_factor=model.E.weight)
    return Tucker(model.core.data, [model.R.weight, model.S.weight, model.O.weight])


def _check_criterion(criterion):
    """The fused loss kind ("bce" or "ce") a criterion selects; TypeError for anything the kernels do not implement."""
    if criterion is None:
        return "bce"
    if isinstance(criterion, nn.BCELoss) and criterion.reduction == "mean":
        return "bce"
    if (isinstance(criterion, nn.CrossEntropyLoss) and criterion.reduction == "mean" and criterion.weight is None
            and criterion.ignore_index == -100 and criterion.label_smoothing == 0.0):
        return "ce"
    raise TypeError("the fused path implements nn.BCELoss(reduction='mean') (train.py:136) and "
                    "nn.CrossEntropyLoss(reduction='mean') without weight, ignore_index or label_smoothing "
                    "(the smoothing comes from the loader); got %r" % (criterion,))


def _relation_batches(loader):
    """Relation batches without end: the loader restarts (a new permutation) whenever it runs out."""
    while True:
        empty = True
        for batch in loader:
            empty = False
            yield batch
        if empty:
            raise ValueError("relation_loader yields no batches")


def train_one_epoch(model, optimizer, criterion, train_loader, regularization_coeff=1e-4, relation_loader=None,
                    relation_weight=0.0):
    """One pass over ``train_loader``; returns (mean loss, mean ||rgrad||) like train.py:91.

    ``relation_loader`` (a DeviceEpoch over data.relation_train_dataset) adds the relation-prediction term with weight
    ``relation_weight`` to every step (optim.RelationTerm; the loss then includes it): each step draws the loader's next
    (s, o) batch, restarting it when it runs out.  The return value is then (mean loss, mean ||rgrad||, mean relation
    cross-entropy), the last None when the weight is 0 (nothing of the term runs)."""
    loss_kind = _check_criterion(criterion)
    relation_weight = float(relation_weight)
    if not (relation_weight >= 0.0 and relation_weight != float("inf")):
        raise ValueError(f"relation_weight must be finite and >= 0, got {relation_weight}")
    if relation_loader is None and relation_weight != 0.0:
        raise ValueError("relation_weight > 0 needs a relation_loader")
    model.train()
    device = model.core.device
    n_batches = len(train_loader)
    train_loss = torch.zeros((), device=device)
    train_grad_norm = torch.zeros((), device=device)
    rel_batches = _relation_batches(relation_loader) if relation_loader is not None else None
    rel_loss = torch.zeros((), device=device) if rel_batches is not None and relation_weight > 0 else None
    for features, targets in train_loader:
        score_fn = model(features[:, 0], features[:, 1])
        relation = None
        if rel_batches is not None:
            pairs, rel_targets = next(rel_batches)
            relation = RelationTerm(pairs, rel_targets, relation_weight, relation_loader.label_smoothing)
        loss_fn = FusedLoss(score_fn, targets, train_loader.label_smoothing, regularization_coeff, loss=loss_kind,
                            relation=relation)
        x_k = extract_tensor(model)
        grad_norm = optimizer.fit(loss_fn, x_k)
        optimizer.step()
        train_grad_norm += grad_norm.detach()
        train_loss += optimizer.loss.detach()
        if rel_loss is not None:
            rel_loss += optimizer.rel_loss.detach()
        optimizer.zero_grad(set_to_none=True)
    if relation_loader is None:
        return train_loss.item() / n_batches, train_grad_norm.item() / n_batches      # the epoch's only host sync
    return (train_loss.item() / n_batches, train_grad_norm.item() / n_batches,
            rel_loss.item() / n_batches if rel_loss is not None else None)


@torch.no_grad()
def evaluate(model, criterion, dataloader, n_begin=0, group=None, space="prob"):
    """Filtered ranking + loss over ``dataloader`` (features (s, r, o), targets = filter lists over all splits);
    returns (metrics dict, mean batch loss) like train.py:124-125.  space="prob" (the default): probability-space
    ranks and the reference's BCE, whichever criterion trained the model; space="logit": logit-space ranks and the
    cross-entropy of the un-smoothed filter lists (evaluation.py), comparable with the CE training loss."""
    _check_criterion(criterion)
    _check_space(space, ("prob", "logit"))
    model.eval()
    device = model.core.device
    point = extract_tensor(model)
    n_ent = dataloader.n_entities
    sums = None
    val_loss = torch.zeros(1, dtype=torch.float64, device=device)
    denom = 0
    for features, filters in dataloader:
        ranks, bl, _ = rank_batch(point, features, filters, n_begin, group, space)
        s = _sums_from_ranks(ranks)
        sums = s if sums is None else {k: sums[k] + s[k] for k in s}
        if space == "logit":
            val_loss += bl / features.shape[0]              # cross_entropy(mean) of the batch
        else:
            val_loss += bl / (features.shape[0] * n_ent)    # BCELoss(mean) of the batch (train.py:113)
        denom += features.shape[0]
    n_batches = len(dataloader)
    metrics = {k: v.item() / denom for k, v in sums.items()}
    return metrics, (val_loss / n_batches).float()


def train(model, optimizer, train_loader, val_loader, test_loader, config, regulizer, scheduler=None, log_fn=None,
          start_epoch=None, num_epoches=None, history=None, criterion=None, eval_space="prob", rank_schedule=None,
          relation_loader=None, relation_weight=0.0):
    """train.py:128-167: evaluate once, then per epoch: regulariser step, train epoch, validate, test, snapshot
    (now with the optimiser state), scheduler step.  ``config`` needs ``train_cfg.num_epoches`` and
    ``train_cfg.checkpoint_path`` (configs/base_config.py); ``log_fn(record)`` replaces wandb_log.  ``criterion``:
    the training objective, ``nn.BCELoss(reduction="mean")`` (the reference's, the default) or
    ``nn.CrossEntropyLoss(reduction="mean")`` (see the module docstring).  ``eval_space``: the ``space`` of
    ``evaluate`` ("prob", the default: BCE and probability ranks whichever the criterion; "logit"); each record
    names it.  ``rank_schedule``: {epoch: (r0, r1, r2)}; ``rank.set_rank(model, rank, optimizer)`` runs at the start of
    that epoch (truncation or growth; the optimiser's momentum restarts, the scheduler is untouched).  Each record
    names the rank the epoch trained at.  ``relation_loader`` / ``relation_weight``: the relation-prediction term of
    train_one_epoch; each record then carries its mean (``train_rel_loss``)."""
    criterion = nn.BCELoss(reduction="mean") if criterion is None else criterion
    _check_criterion(criterion)
    _check_space(eval_space, ("prob", "logit"))
    num_epoches = num_epoches if num_epoches is not None else config.train_cfg.num_epoches
    start_epoch = start_epoch if start_epoch is not None else 1
    history = history if history is not None else []
    prev_val_mrr = evaluate(model, criterion, val_loader, space=eval_space)[0]["mrr"]
    state = None
    for epoch in range(start_epoch, num_epoches + start_epoch):
        if rank_schedule and epoch in rank_schedule:
            set_rank(model, rank_schedule[epoch], optimizer)
        regularization_coeff = regulizer.step()
        t0 = time.perf_counter()
        rel = {}
        if relation_loader is None:
            train_loss, train_norm = train_one_epoch(model, optimizer, criterion, train_loader,
                                                     regularization_coeff=regularization_coeff)
        else:
            train_loss, train_norm, rel["train_rel_loss"] = train_one_epoch(
                model, optimizer, criterion, train_loader, regularization_coeff=regularization_coeff,
                relation_loader=relation_loader, relation_weight=relation_weight)
        epoch_time = time.perf_counter() - t0
        val_metrics, val_loss = evaluate(model, criterion, val_loader, space=eval_space)
        t0 = time.perf_counter()
        test_metrics, test_loss = evaluate(model, criterion, test_loader, space=eval_space)
        torch.cuda.synchronize()
        eval_time = time.perf_counter() - t0
        record = dict(epoch=epoch, train_loss=train_loss, grad_norm=train_norm, val_loss=float(val_loss),
                      test_loss=float(test_loss), lr=optimizer.param_groups[0]["lr"], reg_coeff=regularization_coeff,
                      epoch_time=epoch_time, eval_time=eval_time, eval_space=eval_space, rank=list(model.core.shape),
                      **rel,
                      **{"val_" + k: v for k, v in val_metrics.items()},
                      **{"test_" + k: v for k, v in test_metrics.items()})
        history.append(record)
        path = getattr(config.train_cfg, "checkpoint_path", None)
        if path:
            state = checkpoint.save(os.path.join(path, "snapshot.pth"), model, optimizer, scheduler, epoch, history)
            if val_metrics["mrr"] - prev_val_mrr > 5e-4:
                prev_val_mrr = val_metrics["mrr"]
                checkpoint.save(os.path.join(path, f"rk_{model.rank[1]}_{epoch}.pth"), model, optimizer, scheduler,
                                epoch, history)
        if scheduler is not None:
            scheduler.step()
        if log_fn is not None:
            log_fn(record)
    return history if state is None else state
