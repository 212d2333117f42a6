"""Quality run on the REAL WN18RR triples through the package's own epoch driver (rtucker_b200.train = the reference's
train.py:69-167), rank (10, 200, 200), batch 512, rsgd momentum 0.8, label smoothing 0.1, seed 322, with either
  --recipe head    what the reference's HEAD runs: OneCycleLR(max_lr=600, total_steps=500, pct_start=0.2, div_factor=5.5,
                   linear) stepped per epoch (train.py:213-215), regulariser 1e-11 -> 1e-16 linear in 500 steps
                   (configs/base_config.py:12-21)
  --recipe readme  README.md:36-45: lr 2000 x 0.9981^epoch, regulariser "exp" 1e-4 -> 3e-9 in 350 steps (with HEAD's
                   unit-normalised step this recipe oscillates X <-> -X while reg * ||T||^2 dominates the loss, SURVEY
                   App. B.6: the loss then only follows the regulariser's decay)

    python tools/train_wn18rr.py --epochs 150 --variant 2 --out profiles/r02_train_wn18rr_v2.json

Writes one JSON record per epoch (train loss, ||rgrad||, validation / test MRR and Hits@k, epoch seconds).
--eval-space logit adds, next to those (which stay the probability-space ones), per split: the logit-space metrics
(<split>_logit_mrr, ...), the cross-entropy evaluation loss (<split>_ce_loss) and the number of queries whose target
ties with an unfiltered entity (equal > 0) in each space (<split>_ties_prob, <split>_ties_logit).  The score
kernel variant 2 (fp16-operand tcgen05) and variant 0 (fp32 FFMA, the 1e-5 parity path) are run on identical seeds
and batches (host shuffle = the reference's RandomSampler draw) so that their curves can be compared point by point.
"""
import argparse
import json
import math
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rtucker_b200 import asymmetric, symmetric                      # noqa: E402
from rtucker_b200 import train as T                                  # noqa: E402
from rtucker_b200.data import DeviceEpoch, datasets_from_ids, wn18rr_fixture   # noqa: E402
from rtucker_b200.evaluation import rank_batch                      # noqa: E402


class LinearRegulariser:
    """SimpleDecreasingPolicy(strategy="linear") (src/utils/regularization.py:22-52)."""

    def __init__(self, base, final, steps):
        self.val, self.final, self.d = base, final, (base - final) / steps

    def step(self):
        if self.val > self.final:
            self.val -= self.d
        return self.val


class ExpRegulariser:
    """SimpleDecreasingPolicy(strategy="exp") of the reference (src/utils/regularization.py:22-52): multiply by
    (final / base)^(1 / num_steps) per step until the final value is reached."""

    def __init__(self, base, final, steps):
        self.val, self.final, self.q = base, final, math.pow(final / base, 1.0 / steps)

    def step(self):
        if self.val > self.final:
            self.val *= self.q
        return self.val


@torch.no_grad()
def tie_census(model, loader):
    """Queries of ``loader`` whose target ties with at least one unfiltered entity, in probability and logit space."""
    point = T.extract_tensor(model)
    ties = {"prob": 0, "logit": 0}
    for features, filters in loader:
        for space in ties:
            ties[space] += int((rank_batch(point, features, filters, space=space)[2][1] > 0).sum())
    return ties


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=100)
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--mode", default="asymmetric", choices=["asymmetric", "symmetric"])
    ap.add_argument("--seed", type=int, default=322)
    ap.add_argument("--lr", type=float, default=2000.0)
    ap.add_argument("--lr-decay", type=float, default=0.9981)
    ap.add_argument("--eval-every", type=int, default=5)
    ap.add_argument("--recipe", default="head", choices=["head", "readme"])
    ap.add_argument("--total-epochs", type=int, default=500, help="length of the HEAD recipe's one-cycle schedule")
    ap.add_argument("--loss", default="bce", choices=["bce", "ce"],
                    help="training objective: the reference's label-smoothed BCE or the 1-N softmax cross-entropy "
                         "(evaluation reports the BCE and the filtered ranks either way)")
    ap.add_argument("--eval-space", default="prob", choices=["prob", "logit"],
                    help="logit: also report logit-space ranks, the cross-entropy evaluation loss and tie counts")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    ids = wn18rr_fixture()
    assert ids is not None, "tests/golden/wn18rr_ids.npz is missing"
    train_ds, valid_ds, test_ds = datasets_from_ids(ids, label_smoothing=0.1)
    rank = (10, 200, 200)
    torch.manual_seed(args.seed)
    mod = asymmetric if args.mode == "asymmetric" else symmetric
    model = mod.R_TuckER((ids["n_entities"], ids["n_relations"]), rank)
    model.init(None)
    model.to(dev)
    params = [model.core, model.S.weight, model.R.weight, model.O.weight] if args.mode == "asymmetric" else \
        [model.core, model.E.weight, model.R.weight]
    opt = mod.RSGDwithMomentum(params, rank, args.lr, 0.8, score_variant=args.variant, use_graphs=True)
    if args.recipe == "readme":
        sched = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=args.lr_decay)
        reg = ExpRegulariser(1e-4, 3e-9, 350)
    else:
        sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=600, total_steps=args.total_epochs,
                                                    pct_start=100 / args.total_epochs, div_factor=5.5,
                                                    cycle_momentum=False, anneal_strategy="linear")
        reg = LinearRegulariser(1e-11, 1e-16, 500)
    train_loader = DeviceEpoch(train_ds, 512, dev, shuffle="host", drop_last=True)
    val_loader = DeviceEpoch(valid_ds, 512, dev, shuffle=False)
    test_loader = DeviceEpoch(test_ds, 512, dev, shuffle=False)
    crit = torch.nn.CrossEntropyLoss(reduction="mean") if args.loss == "ce" else torch.nn.BCELoss(reduction="mean")
    hist = []
    t_start = time.perf_counter()
    for epoch in range(1, args.epochs + 1):
        r = reg.step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss, gnorm = T.train_one_epoch(model, opt, crit, train_loader, regularization_coeff=r)
        torch.cuda.synchronize()
        rec = dict(epoch=epoch, train_loss=loss, grad_norm=gnorm, lr=opt.param_groups[0]["lr"], reg=r,
                   epoch_s=time.perf_counter() - t0)
        if epoch % args.eval_every == 0 or epoch == 1 or epoch == args.epochs:
            t0 = time.perf_counter()
            vm, vl = T.evaluate(model, crit, val_loader)
            tm, tl = T.evaluate(model, crit, test_loader)
            torch.cuda.synchronize()
            # orthonormality of the factors (the retraction assumes U^T U = I and never re-orthonormalises): max |U^T U - I|
            defect = {}
            for name, prm in model.named_parameters():
                if prm.dim() == 2:
                    U = prm.data.double()
                    defect[name] = float((U.T @ U - torch.eye(U.shape[1], dtype=U.dtype, device=U.device)).abs().max())
            rec.update(ortho_defect=defect)
            rec.update(eval_s=time.perf_counter() - t0, val_loss=float(vl), test_loss=float(tl),
                       **{"val_" + k: v for k, v in vm.items()}, **{"test_" + k: v for k, v in tm.items()})
            if args.eval_space == "logit":
                for split, loader in (("val", val_loader), ("test", test_loader)):
                    lm, ll = T.evaluate(model, crit, loader, space="logit")
                    ties = tie_census(model, loader)
                    rec.update({f"{split}_logit_{k}": v for k, v in lm.items()})
                    rec.update({f"{split}_ce_loss": float(ll), f"{split}_ties_prob": ties["prob"],
                                f"{split}_ties_logit": ties["logit"], f"{split}_queries": len(loader.dataset)})
        if not (args.recipe == "head" and epoch >= args.total_epochs):
            sched.step()
        hist.append(rec)
        print(json.dumps(rec), flush=True)
    summary = dict(config=dict(dataset="WN18RR (real triples, tests/golden/wn18rr_ids.npz)", mode=args.mode, rank=rank,
                               batch=512, optim="rsgd", recipe=args.recipe,
                               momentum=0.8, label_smoothing=0.1, seed=args.seed, score_variant=args.variant,
                               loss=args.loss, eval_space=args.eval_space,
                               device=torch.cuda.get_device_name(dev), power_limit_w=_power_limit(),
                               epochs=args.epochs, steps_per_epoch=len(train_loader)),
                   wall_s=time.perf_counter() - t_start, history=hist)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f)


def _power_limit():
    """The card's power limit in W, read next to the measurement (None where nvidia-smi is not available)."""
    import subprocess
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        return None


if __name__ == "__main__":
    main()
