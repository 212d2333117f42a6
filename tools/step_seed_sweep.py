"""The errors test_step_parity bounds, for its huge-step configurations over many problem seeds, and, for any step
over a bound, which small-stage call deviates from its fp64 restatement (tests/cpu_ops.SmallStage).

    python tools/step_seed_sweep.py [--seeds 40] [--out sweep.json]

Each draw builds the configuration's problem from torch.Generator().manual_seed(seed) instead of the name-derived
seed of the test, takes the test's steps, and prints per step every quantity the test bounds: the relative errors of
loss, ||rgrad|| and the probed point against the fp64 analytic oracle re-seeded from the device state (1e-5), the
point and ||rgrad|| against the free-running oracle (1e-3), and the orthonormality defect of the factors (5e-6).
The small stage's calls of an over-bound step are recorded (inputs and outputs, on the host) and replayed through the oracle: the report gives
each call's largest per-tile relative error and the relative gap at r of the retraction's unfolding Grams.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import cpu_ops                       # noqa: E402
import small_stage_checks as chk     # noqa: E402
from test_gpu_step import CONFIGS, make_batch, ortho, probes   # noqa: E402

f64 = torch.float64
BOUNDS = {"loss": 1e-5, "norm": 1e-5, "point": 1e-5, "traj_point": 1e-3, "traj_norm": 1e-3, "ortho": 5e-6}
CALLS = ("prepare", "grad", "norm", "project", "retract")


def _host(x):
    if torch.is_tensor(x):
        return x.detach().cpu().clone()
    if isinstance(x, (list, tuple)):
        return type(x)(_host(y) for y in x)
    return x


class Recorder:
    """Stands in for the engine's ops.SmallStage and keeps host copies of the arguments and results of each call."""

    def __init__(self, inner):
        self.inner, self.calls = inner, []

    def __getattr__(self, name):
        f = getattr(self.inner, name)
        if name not in CALLS:
            return f

        def wrapped(*a, **k):
            ins = _host(a)
            out = f(*a, **k)
            torch.cuda.synchronize()
            self.calls.append((name, ins, _host(out)))
            return out
        return wrapped


def replay(calls, rank, B, sym):
    """Per-call largest tile-relative error of the device outputs against the oracle fed the same inputs."""
    ref = cpu_ops.SmallStage(rank, B, sym, "cpu")
    res = {}
    for name, ins, out in calls:
        if name == "prepare":
            ref.prepare(ins[0])
        elif name == "grad":
            r = ref.grad(*ins)
            res["grad"] = max(chk.tile_relerr(o, x) for o, x in zip(out, r))
        elif name == "norm":
            hyper = ins[4].clone()
            adam = ins[5].clone() if len(ins) > 5 and ins[5] is not None else None
            r = ref.norm(*ins[:4], hyper, adam=adam)
            res["norm"] = max(chk.tile_relerr(o, x) for o, x in zip(out, r))
        elif name == "project":
            pS, K, L = ref.project(*ins)
            res["project"] = max([chk.tile_relerr(out[0], pS)] + [chk.tile_relerr(a, b) for a, b in zip(out[1] + out[2], K + L)])
        elif name == "retract":
            spectra = []
            core_new, Z1, Z2, _ = ref.retract(*ins[:6], spectra=spectra)
            gaps = [chk.relgap(spectra[i], rank[i]) for i in range(3)]
            Zs = [(a, b) for a, b in zip(out[1], out[2])]
            ortho_err = max(float((z1.T @ z1 + z2.T @ g.double() @ z2 - torch.eye(z1.shape[1], dtype=f64)).abs().max())
                            for (z1, z2), g in zip(Zs, [ins[2], ins[3], ins[3] if sym else ins[4]]))
            res["retract"] = {"core_new vs oracle (gauge-dependent)": chk.tile_relerr(out[0], core_new),
                              "relgap": gaps, "orthonormality of Z": ortho_err}
    return res


def run_draw(name, seed, dev):
    import analytic as A
    from rtucker_b200.engine import SparseTargets, StepEngine
    A.ELEMENTWISE_FP32 = True
    _, N, M, rank, B, sym, beta, lr_rel, reg_rel, steps = next(c for c in CONFIGS if c[0] == name)
    g = torch.Generator().manual_seed(seed)
    R, S = ortho(M, rank[0], g), ortho(N, rank[1], g)
    O = S if sym else ortho(N, rank[2], g)
    core = torch.randn(rank, generator=g, dtype=f64) * (3.0 * (N * N * M / (rank[0] * rank[1] * rank[2])) ** 0.5) / 3
    lr, reg = lr_rel * float(core.norm()), reg_rel / float(core.norm()) ** 2
    Pm = torch.nn.Parameter
    pc = Pm(core.float().contiguous().to(dev))
    pf = [Pm(R.float().contiguous().to(dev)), Pm(S.float().contiguous().to(dev))] + ([] if sym else [Pm(O.float().contiguous().to(dev))])
    eng = StepEngine(pc, pf, sym, B, beta)
    free = A.RSGDState(A.Point(core.clone(), [R.clone(), S.clone(), S.clone() if sym else O.clone()], sym), beta)
    rec = Recorder(eng.small)
    eng.small = rec
    three = lambda fs: [fs[0], fs[1], fs[1] if sym else fs[2]]
    out = []
    for it in range(steps):
        rel, sub, off, idx = make_batch(N, M, B, g)
        st = A.RSGDState(A.Point(pc.data.double().cpu(), three([p.data.double().cpu() for p in pf]), sym), beta)
        if beta is not None and eng.has_old:
            st.old = A.Point(eng.core_old.double().cpu(), three([u.double().cpu() for u in eng.U_old]), sym)
            st.direction = A.Tangent(eng.dS_dir_old.double().cpu(), three([v.double().cpu() for v in eng.dV_dir]))
        n_ref = st.fit(rel, sub, off, idx, 0.1, reg)
        x_ref = st.step(lr)
        n_free = free.fit(rel, sub, off, idx, 0.1, reg)
        free.step(lr)
        rec.calls = []
        n_dev = eng.fit(rel.int().to(dev), sub.int().to(dev), SparseTargets(off.int().to(dev), idx.int().to(dev)), 0.1, reg)
        eng.step(lr)
        torch.cuda.synchronize()
        x_dev = A.Point(pc.data.double().cpu(), three([p.data.double().cpu() for p in pf]), sym)
        pr = probes(x_ref, torch.Generator().manual_seed(it))
        row = {"step": it,
               "loss": abs(float(eng.loss.cpu()) - float(st.loss)) / abs(float(st.loss)),
               "norm": abs(float(n_dev.cpu()) - float(n_ref)) / float(n_ref),
               "point": float((pr(x_dev) - pr(x_ref)).norm() / pr(x_ref).norm()),
               "traj_point": float((pr(x_dev) - pr(free.x)).norm() / pr(free.x).norm()),
               "traj_norm": abs(float(n_dev.cpu()) - float(n_free)) / float(n_free),
               "ortho": max(float((p.data.double().T @ p.data.double() - torch.eye(p.shape[1], dtype=f64, device=dev)).abs().max())
                            for p in pf)}
        row["over"] = [k for k, b in BOUNDS.items() if row[k] > b]
        if row["over"]:
            row["small_stage"] = replay(rec.calls, rank, B, sym)
        out.append(row)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--seeds", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("step_seed_sweep: needs a CUDA device")
    dev = torch.device("cuda:0")
    report = {"device": torch.cuda.get_device_name(0), "draws": []}
    for name in ("huge-step-asym", "huge-step-sym"):
        for seed in range(args.seeds):
            rows = run_draw(name, seed, dev)
            print(f"{name:16s} seed {seed:2d}  " + "  ".join(
                f"[{r['step']}] " + " ".join(f"{k} {r[k]:.1e}" for k in BOUNDS) + (f" OVER {r['over']}" if r["over"] else "")
                for r in rows), flush=True)
            for r in rows:
                if "small_stage" in r:
                    print("    step", r["step"], json.dumps(r["small_stage"]), flush=True)
            report["draws"].append({"config": name, "seed": seed, "steps": rows})
    if args.out:
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
