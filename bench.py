#!/usr/bin/env python
"""bench.py -- train triples/s of the R-TuckER hot path (1-N fwd + bwd + RSGD step incl. retraction) and
filtered-eval queries/s (BASELINE.json metric), on the REAL WN18RR triples when the id fixture is present
(tests/golden/wn18rr_ids.npz, written from the reference's data/WN18RR by tests/golden/make_golden.py), else on a
seeded synthetic graph of the same shape.

    python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path (one JSON line)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (port, oracle/)
    torchrun ... bench.py --gpus N ...                       # entity-sharded over NCCL (strong scaling)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/*.npy

A step = one optimiser step (fit + step) on one batch of 512 (s, r) queries.
`value`       triples/s with the batches already resident in HBM (CUDA events around K steps, CUDA graphs).
`e2e`         same metric through the public API (model(...) -> FusedLoss -> optimizer.fit/step) with the batch coming
              from pinned HOST memory every step and the loss read back to the host every step.
`value_strict_fp32`  the same K steps with the fp32 FFMA score kernel (variant 0: 1e-5 parity path).
`roofline`    the kernel FAMILY with the largest share of the step; `roofline_all` lists every family (score GEMMs
              against the tensor peak, tall-skinny passes against HBM, N-independent stage as a latency-bound
              share, query contraction, fused eval), each with its share of ms_per_step.
`cpu_baseline`       the reference's step (oracle/reference_step.py port) on this host's cores, bounded sample.
`torch_gpu_baseline` the same port with CUDA tensors: stock cuBLAS / cuSOLVER / ATen on this very GPU.
`c5`          the synthetic 1M-entity / rank-(200,200,200) workload (BASELINE configs[4]) on the same ranks: the
              curve north_star asks for, recorded by every driver run (1/2/4/8 GPUs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n_entities, n_relations incl. reverse, rank, n_queries, mean objects per query)
    "wn18rr": dict(N=40943, M=22, rank=(10, 200, 200), Q=103509, mean_obj=1.678, sym=False),
    "fb15k237": dict(N=14541, M=474, rank=(200, 20, 20), Q=149689, mean_obj=3.636, sym=False),
    "wn18rr-sym": dict(N=40943, M=22, rank=(10, 200, 200), Q=103509, mean_obj=1.678, sym=True),
    "synthetic-1m": dict(N=1000000, M=1000, rank=(200, 200, 200), Q=200000, mean_obj=5.0, sym=False),
}
BATCH = 512
LABEL_SMOOTHING = 0.1
MOMENTUM = 0.8
LR = 109.09      # OneCycleLR(max_lr=600, div_factor=5.5) at epoch 1 (train.py:213-215)
REG = 1e-11      # configs/base_config.py:19
SEED = 322       # README.md:45
FFMA_PEAK_TF = 148 * 128 * 2 * 1.965e9 / 1e12      # nominal FP32 FFMA peak at the measured max clock (74.4)
DUMP_ROWS = 8192  # entity-factor rows --dump-outputs keeps: whole factors are 65 MB (WN18RR) to 1.6 GB (1M entities)


def synth_graph(w, seed=1234):
    """Seeded synthetic (s,r)->objects vocabulary of the workload's shape (SURVEY.md App. C.4)."""
    rng = np.random.default_rng(seed)
    N, M, Q = w["N"], w["M"], w["Q"]
    pop = 1.0 / np.arange(1, N + 1) ** 0.6
    pop /= pop.sum()
    perm = rng.permutation(N)
    keys = set()
    feats = np.zeros((Q, 2), np.int32)
    n = 0
    while n < Q:
        s = perm[rng.choice(N, size=Q, p=pop)]
        r = rng.integers(0, M, size=Q)
        for a, b in zip(s.tolist(), r.tolist()):
            if (a, b) not in keys:
                keys.add((a, b))
                feats[n] = (a, b)
                n += 1
                if n == Q:
                    break
    extra = rng.geometric(1.0 / w["mean_obj"], size=Q)  # >= 1, mean = mean_obj
    extra = np.minimum(extra, 400)
    off = np.zeros(Q + 1, np.int64)
    np.cumsum(extra, out=off[1:])
    idx = perm[rng.choice(N, size=int(off[-1]), p=pop)].astype(np.int32)
    # unique + ascending per query
    lists = [np.unique(idx[off[i]:off[i + 1]]) for i in range(Q)]
    cnt = np.asarray([len(x) for x in lists], np.int64)
    off = np.zeros(Q + 1, np.int64)
    np.cumsum(cnt, out=off[1:])
    return feats, off, np.concatenate(lists).astype(np.int32), cnt


def batch_arrays(feats, off, idx, cnt, items):
    c = cnt[items]
    boff = np.zeros(len(items) + 1, np.int32)
    np.cumsum(c, out=boff[1:])
    gather = np.repeat(off[items] - boff[:-1], c) + np.arange(int(boff[-1]), dtype=np.int64)
    return feats[items], boff, idx[gather]


def load_workload(name):
    """(w, graph, data_label): graph = (features [Q,2], off, idx, cnt) of the train (s, r) -> objects vocabulary.
    The WN18RR workloads use the real triples through the package's own SparseKGDataset when the fixture exists."""
    w = dict(WORKLOADS[name])
    if name in ("wn18rr", "wn18rr-sym"):
        from rtucker_b200.data import datasets_from_ids, wn18rr_fixture
        ids = wn18rr_fixture()
        if ids is not None:
            train, valid, test = datasets_from_ids(ids, label_smoothing=LABEL_SMOOTHING)
            w["Q"] = len(train)
            w["eval"] = test
            return w, (train.features, train.off, train.idx, train.counts), \
                "real WN18RR train triples (tests/golden/wn18rr_ids.npz, ids of the reference's data/WN18RR)"
    return w, synth_graph(w), "synthetic"


def init_params(w, seed=SEED):
    """R_TuckER.init: xavier core + QR-orthonormalised xavier factors on the CPU generator."""
    from rtucker_b200 import asymmetric, symmetric
    np.random.seed(seed)
    torch.manual_seed(seed)
    mod = symmetric if w["sym"] else asymmetric
    model = mod.R_TuckER((w["N"], w["M"]), w["rank"])
    model.init(None)
    return model


class ClockSampler:
    def __init__(self):
        self.rows, self.proc = [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", os.environ.get("LOCAL_RANK", "0")],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def reference_steps(w, graph, n_steps, warmup, threads=None, device="cpu"):
    """Times the reference's train step (port, oracle/reference_step.py) on the host cores -- or, with
    device="cuda", the same PyTorch code on CUDA tensors (stock cuBLAS / cuSOLVER).  Dense targets are built outside
    the timed region (the reference builds them in DataLoader worker processes)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_step as RS
    if threads:
        torch.set_num_threads(threads)
    feats, off, idx, cnt = graph
    model = init_params(w)
    dev = torch.device(device)
    P = lambda t: t.data.to(dev)  # noqa: E731
    if w["sym"]:
        st = RS.ReferenceStepper(P(model.core), P(model.R.weight), P(model.E.weight), None, None)
    else:
        st = RS.ReferenceStepper(P(model.core), P(model.R.weight), P(model.S.weight), P(model.O.weight), MOMENTUM)
    rng = np.random.default_rng(7)
    order = rng.permutation(len(cnt))
    triples, total = 0, 0.0
    for i in range(warmup + n_steps):
        items = order[i * BATCH:(i + 1) * BATCH]
        f, boff, bidx = batch_arrays(feats, off, idx, cnt, items)
        tg = RS.dense_targets(w["N"], torch.from_numpy(boff.astype(np.int64)), torch.from_numpy(bidx), LABEL_SMOOTHING).to(dev)
        ft = torch.from_numpy(f.astype(np.int64)).to(dev)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        st.train_step(ft[:, 0], ft[:, 1], tg, REG, LR)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if i >= warmup:
            total += dt
            triples += int(cnt[items].sum())
    return triples / total, total / n_steps, torch.get_num_threads()


def metric_name(data_label):
    return "train triples/s (1-N fwd+bwd+RSGD step), WN18RR" + ("" if data_label.startswith("real") else " shape")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w, graph, data_label = load_workload(args.workload)
    # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host core it can get
    tps, sps, cores = reference_steps(w, graph, args.steps, args.warmup, threads=os.cpu_count())
    line = {
        "impl": "reference", "metric": metric_name(data_label),
        "value": tps, "unit": "triples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": data_label,
        "config": config_dict(w, args),
        "cpu_baseline": {"value": tps, "unit": "triples/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} full train steps of B={BATCH} (oracle/reference_step.py), dense targets built outside the timed region"},
        "e2e": {"value": tps, "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel, from the committed ncu --set full capture
    (profiles/ncu_traffic.json); None if never captured."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.isfile(path):
        return json.load(open(path)).get(key)
    return None


def config_dict(w, args):
    return {"workload": f"{args.workload}: N={w['N']} entities, M={w['M']} relations, "
                        f"rank={tuple(w['rank'])}, batch {BATCH}, {'SF-Tucker rgd' if w['sym'] else 'Tucker rsgd'} "
                        f"beta={MOMENTUM}, label_smoothing={LABEL_SMOOTHING}, lr={LR}, reg={REG}, init seed {SEED}",
            "l2": "per-step working set (factors + tangent/momentum buffers) > 126 MB L2; no explicit flush"}


class Runner:
    """One model + optimiser of a workload on this rank's entity shard, with pre-assembled batches."""

    def __init__(self, w, graph, dev, world, rank, group, variant, use_graphs, n_batches):
        from rtucker_b200 import asymmetric, symmetric
        self.w, self.dev, self.world, self.group = w, dev, world, group
        feats, off, idx, cnt = graph
        model = init_params(w)
        N = w["N"]
        per = (N + world - 1) // world
        self.n_begin, self.n_end = rank * per, min(N, (rank + 1) * per)
        with torch.no_grad():
            if w["sym"]:
                model.E.weight.data = model.E.weight.data[self.n_begin:self.n_end].contiguous()
            else:
                model.S.weight.data = model.S.weight.data[self.n_begin:self.n_end].contiguous()
                model.O.weight.data = model.O.weight.data[self.n_begin:self.n_end].contiguous()
        self.model = model.to(dev)
        mod = symmetric if w["sym"] else asymmetric
        kw = dict(group=group, n_total=N, n_begin=self.n_begin, score_variant=variant, use_graphs=use_graphs)
        if w["sym"]:
            self.opt = mod.RGD([model.core, model.E.weight, model.R.weight], w["rank"], LR, **kw)
        else:
            self.opt = mod.RSGDwithMomentum([model.core, model.S.weight, model.R.weight, model.O.weight], w["rank"], LR,
                                            MOMENTUM, **kw)
        self.opt.param_groups[0]["lr"] = LR
        rng = np.random.default_rng(7)
        order = rng.permutation(len(cnt))
        self.host_batches, self.triples = [], []
        for i in range(n_batches):
            items = order[(i * BATCH) % (len(order) - BATCH):][:BATCH]
            f, boff, bidx = batch_arrays(feats, off, idx, cnt, items)
            self.host_batches.append([torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (f, boff, bidx)])
            self.triples.append(int(cnt[items].sum()))

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def one_step(self, fd, od, xd):
        from rtucker_b200.engine import SparseTargets
        from rtucker_b200.optim import FusedLoss
        score_fn = self.model(fd[:, 0], fd[:, 1])
        self.rgrad_norm = self.opt.fit(FusedLoss(score_fn, SparseTargets(od, xd), LABEL_SMOOTHING, REG), None)
        self.opt.step()

    def max_over_ranks(self, ms):
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    def timed_resident(self, warmup, steps):
        """K steps on batches already in HBM; returns (ms total = max over ranks, triples)."""
        dev_batches = [[t.to(self.dev) for t in hb] for hb in self.host_batches[:warmup + steps]]
        for i in range(warmup):
            self.one_step(*dev_batches[i])
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(warmup, warmup + steps):
            self.one_step(*dev_batches[i])
        e1.record()
        self.barrier()
        self.dev_batches = dev_batches
        return self.max_over_ranks(e0.elapsed_time(e1)), sum(self.triples[warmup:warmup + steps])

    def dump_outputs(self, out_dir):
        """What the last step returned to its caller, as out_dir/<name>.npy (float32): the loss and ||rgrad|| of fit(),
        the core and relation factor after step(), and of every entity factor the rows of a fixed seeded sample of
        DUMP_ROWS global row ids (ascending; the same rows on any number of GPUs).  Written by rank 0."""
        w, model = self.w, self.model
        rows = np.sort(np.random.default_rng(SEED).choice(w["N"], size=min(w["N"], DUMP_ROWS), replace=False))
        out = {"loss": self.opt.loss, "rgrad_norm": self.rgrad_norm, "core": model.core.data, "R": model.R.weight.data}
        mine = (rows >= self.n_begin) & (rows < self.n_end)
        for name in ("E",) if w["sym"] else ("S", "O"):
            local = getattr(model, name).weight.data
            sample = torch.zeros(len(rows), local.shape[1], dtype=local.dtype, device=self.dev)
            sample[torch.from_numpy(np.flatnonzero(mine)).to(self.dev)] = \
                local[torch.from_numpy(rows[mine] - self.n_begin).to(self.dev)]
            if self.world > 1:
                torch.distributed.all_reduce(sample)      # each row lives on one rank, the others add zeros
            out[name] = sample
        out = {k: v.detach().cpu().numpy() for k, v in out.items()}
        assert sum(a.nbytes for a in out.values()) <= 64 << 20, "dump exceeds 64 MB: lower DUMP_ROWS"
        if int(os.environ.get("RANK", "0")) == 0:
            os.makedirs(out_dir, exist_ok=True)
            for name, a in out.items():
                np.save(os.path.join(out_dir, name + ".npy"), a)

    def timed_e2e(self, first, steps):
        h2d = d2h = 0
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(first, first + steps):
            hb = self.host_batches[i]
            db = [t.to(self.dev, non_blocking=True) for t in hb]
            h2d = sum(t.numel() * t.element_size() for t in hb)
            self.one_step(*db)
            loss_host = self.opt.loss.cpu()       # device -> host read of the step's result
            d2h = loss_host.numel() * loss_host.element_size()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)), sum(self.triples[first:first + steps]), h2d, d2h

    def eval_qps(self, n_batches, eval_ds=None):
        """Filtered evaluation (fused score + rank) queries/s: the real test split when available, else the train
        queries with their first known object as the target."""
        from rtucker_b200.engine import SparseTargets
        from rtucker_b200.evaluation import rank_batch
        from rtucker_b200.train import extract_tensor
        point = extract_tensor(self.model)
        ebs = []
        for i in range(n_batches):
            if eval_ds is not None:
                f3, boff, bidx = eval_ds.host_batch(np.arange(i * BATCH, min((i + 1) * BATCH, len(eval_ds))))
                f3, boff, bidx = (torch.from_numpy(np.ascontiguousarray(a)) for a in (f3, boff, bidx))
            else:
                f, boff, bidx = self.host_batches[i]
                f3 = torch.cat([f, bidx[boff[:-1].long()][:, None]], dim=1).contiguous()
            ebs.append((f3.to(self.dev), SparseTargets(boff.to(self.dev), bidx.to(self.dev))))
        rank_batch(point, ebs[0][0], ebs[0][1], self.n_begin, self.group)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for f3, flt in ebs:
            rank_batch(point, f3, flt, self.n_begin, self.group)
        e1.record()
        self.barrier()
        ms = self.max_over_ranks(e0.elapsed_time(e1))
        return sum(b[0].shape[0] for b in ebs) / (ms * 1e-3), ms / len(ebs)


def time_score_kernel(run, dev, variant, steps, large):
    """The fused score kernel on its own, launched back to back on the step's inputs (CUDA events on the launching
    stream; its working set -- O, packed images, dO, per-CTA H partials -- exceeds the L2)."""
    from rtucker_b200 import lib, ops as _ops
    w = run.w
    fd, od, xd = run.dev_batches[0]
    model = run.model
    O_fac = model.E.weight.data if w["sym"] else model.O.weight.data
    S_fac = model.E.weight.data if w["sym"] else model.S.weight.data
    B_, r2_ = BATCH, w["rank"][2]
    r_rows = _ops.gather_rows(model.R.weight.data, fd[:, 1].contiguous())
    s_rows = _ops.gather_rows(S_fac, fd[:, 0].contiguous(), run.n_begin)
    if run.world > 1:
        torch.distributed.all_reduce(s_rows)
    qq = _ops.query_fwd(model.core.data, r_rows, s_rows)
    outs = (torch.empty(1, dtype=torch.float64, device=dev), torch.empty(B_, r2_, device=dev), torch.empty_like(O_fac))
    v = variant
    if v == 2 and not _ops.score_v3_supported(r2_):
        v = 1
    if v == 3 and not _ops.score_tc3_supported(B_, O_fac.shape[0], r2_):
        v = 0
    ws_bytes = lib().rt_score_bce_tc3_ws_bytes(B_, O_fac.shape[0], r2_) if v == 3 else \
        lib().rt_score_bce_ws_bytes(B_, O_fac.shape[0], r2_, v)
    ws_s = torch.empty(int(ws_bytes) + 16, dtype=torch.uint8, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def run_score(phases=7):
        _ops.score_bce_fwd_bwd(qq, None if v >= 2 else qq, O_fac, od, xd, LABEL_SMOOTHING, n_total=w["N"], b_total=B_,
                               n_begin=run.n_begin, variant=v, out=outs, ws=ws_s, o_absmax=1.0 if v == 2 else None,
                               phases=phases)
    reps = max(10, steps)

    def timed(phases):
        for _ in range(3):
            run_score(phases)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            run_score(phases)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    run_score(7)
    out = {"variant": v, "op_ms": timed(7), "kernel_ms": timed(2) if v == 2 else None, "launches_timed": reps, "large": None}
    if large and v == 2:
        try:
            N1, r1m = 1000000, 200
            O1 = torch.randn(N1, r1m, device=dev) * (1.0 / N1 ** 0.5)
            q1 = torch.randn(B_, r1m, device=dev) * 4.0 * (N1 / r1m) ** 0.5      # logits ~ N(0, 4^2)
            out1 = (torch.empty(1, dtype=torch.float64, device=dev), torch.empty(B_, r1m, device=dev), torch.empty_like(O1))
            ws1 = torch.empty(int(lib().rt_score_bce_ws_bytes(B_, N1, r1m, 2)) + 16, dtype=torch.uint8, device=dev)

            def run1(phases=7):
                _ops.score_bce_fwd_bwd(q1, None, O1, od, xd, LABEL_SMOOTHING, n_total=N1, b_total=B_, variant=2,
                                       out=out1, ws=ws1, o_absmax=1.0, phases=phases)
            run1(7)
            for _ in range(2):
                run1(2)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(5):
                run1(2)
            e1.record()
            torch.cuda.synchronize()
            out["large"] = {"kernel_ms": e0.elapsed_time(e1) / 5, "flops": 6.0 * B_ * N1 * r1m, "launches_timed": 5}
            del O1, out1, ws1
        except RuntimeError as exc:      # out of memory on a smaller part: the number is simply absent
            out["large"] = {"error": str(exc)[:120]}
    return out


def rooflines(w, n_local, ms_step, stage_ms, score_timing, eval_ms, peaks, small_flops=None):
    """One entry per kernel family (SURVEY.md section 8d), each with its share of the step."""
    r0, r1, r2 = w["rank"]
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    tf_burst = float(peaks.get("bf16_tflops", 1590.0))
    src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
    st = stage_ms
    tot_eager = sum(st.values()) or 1.0
    share = lambda keys: sum(st.get(k, 0.0) for k in keys) / tot_eager  # noqa: E731
    out = []
    # (b) fused score + BCE + backward
    flops_b = 6.0 * BATCH * n_local * r2
    k_ms = (score_timing or {}).get("kernel_ms") or (score_timing or {}).get("op_ms") or st.get("score_bce_fwd_bwd")
    ach = flops_b / (k_ms * 1e-3) / 1e12 if k_ms else None
    vnt = (score_timing or {}).get("variant", 0)
    # variant 3 spends 3 TF32 MMAs (half the bf16 rate) per product: its roofline is bf16 peak / 6
    peak_b = (tf_burst / 6.0) if vnt == 3 else (tf_burst if vnt else FFMA_PEAK_TF)
    entry_b = {"family": "b: fused 1-N score + BCE + backward (variant %d)" % vnt, "bound": "tensor", "achieved": ach,
               "peak": peak_b, "unit": "TFLOP/s", "frac": ach / peak_b if ach else None,
               "peak_source": (src + " bf16_tflops / 6 (fp32-accurate products = 3 TF32 MMAs at half the bf16 rate; op timed alone)") if vnt == 3 else
                              ((src + " bf16_tflops (burst: kernel timed alone)") if vnt else "nominal FP32 FFMA (148 SMs x 128 lanes x 2 x 1.965 GHz)"),
               "algorithmic_flops_per_launch": flops_b, "ms_per_launch": k_ms, "traffic": ncu_traffic("score_v3:wn18rr" if vnt == 2 else "score_variant%d:wn18rr" % vnt),
               "share_of_step": share(["score_bce_fwd_bwd"]), "timing": score_timing}
    if score_timing and score_timing.get("large") and score_timing["large"].get("kernel_ms"):
        lg = score_timing["large"]
        a1 = lg["flops"] / (lg["kernel_ms"] * 1e-3) / 1e12
        entry_b["same_kernel_on_1m_entities"] = {"ms_per_launch": lg["kernel_ms"], "achieved": a1, "frac": a1 / tf_burst,
                                                 "unit": "TFLOP/s", "algorithmic_flops_per_launch": lg["flops"]}
    out.append(entry_b)
    # (c) tall-skinny passes: HBM roofline, 24 N r bytes per big factor and step (SURVEY 8d)
    big = [r for r in ((r1, r2) if not w["sym"] else (r1,))]
    bytes_c = sum(24.0 * n_local * r for r in big)
    ts_keys = ["tall_skinny_fit", "retract_gram", "retract_apply", "write_back"]
    ms_c = sum(st.get(k, 0.0) for k in ts_keys) - st.get("small_project", 0.0)
    ach_c = bytes_c / (ms_c * 1e-3) / 1e9 if ms_c > 0 else None
    # the same passes as arithmetic: 13 N x r x r products (gradient 3, momentum 6, retraction 4) on tcgen05 as 3 TF32
    # MMAs each, and 4 exact Grams (upper triangle) on the fp64 tensor cores
    n_terms = 13 if not w["sym"] else 7
    n_grams = 4 if not w["sym"] else 2
    rr = float(big[0])
    flops_apply = n_terms * 2.0 * n_local * rr * rr
    flops_gram = n_grams * 2.0 * n_local * rr * (rr + 1) / 2
    tf32_3x_peak = tf_burst / 2.0 / 3.0
    t_floor_ms = (flops_apply / (tf32_3x_peak * 1e12) + flops_gram / 45e12) * 1e3
    out.append({"family": "c: tall-skinny projection / transport / retraction passes (N x r x r)", "bound": "hbm",
                "achieved": ach_c, "peak": hbm, "unit": "GB/s", "frac": ach_c / hbm if ach_c else None,
                "peak_source": src + " hbm_gbs", "algorithmic_bytes_per_step": bytes_c, "ms_per_step": ms_c,
                "traffic": ncu_traffic("tall_skinny:wn18rr"), "share_of_step": ms_c / tot_eager,
                "timing_note": "sum of the N-sized stages of stage_ms (CUDA events)",
                "arithmetic_view": {
                    "note": "at r = 200 these passes are arithmetic-bound at fp32 accuracy, not HBM-bound: fp32-accurate "
                            "products cost 3 TF32 MMAs each (peak = bf16 peak / 2 / 3), the Cholesky of the retraction needs an "
                            "exactly accumulated Gram (fp64 tensor cores, 45 TFLOP/s nominal)",
                    "flops_products_per_step": flops_apply, "flops_grams_per_step": flops_gram,
                    "floor_ms": t_floor_ms, "frac_of_floor": t_floor_ms / ms_c if ms_c > 0 else None}})
    # (c-small) N-independent stage
    sm_keys = ["small_prepare", "small_grad", "small_project", "small_retract_hosvd"]
    # fp64 tensor-core ceiling measured on this part (tools/dmma_probe.cu, profiles/r02_dmma_probe.txt): DMMA m8n8k4 from
    # registers 36.4 TFLOP/s; the plain fp64 pipe delivers 2.9
    DMMA_PEAK_TF = 36.4
    ms_small = sum(st.get(k, 0.0) for k in sm_keys)
    ach_s = small_flops / (ms_small * 1e-3) / 1e12 if (small_flops and ms_small > 0) else None
    out.append({"family": "c-small: N-independent fp64 stage (Gram inverses, projection cores, HOSVD subspaces)",
                "bound": "fp64-tensor", "achieved": ach_s, "peak": DMMA_PEAK_TF, "unit": "TFLOP/s",
                "frac": ach_s / DMMA_PEAK_TF if ach_s else None, "traffic": None,
                "peak_source": "DMMA m8n8k4 throughput measured on this B200 (tools/dmma_probe.cu; nominal fp64 tensor 40 TFLOP/s)",
                "algorithmic_flops_per_step": small_flops, "ms_per_step": ms_small, "share_of_step": share(sm_keys),
                "note": "achieved = fp64 flops of the executor's GEMM operations (2 m n K, half for a symmetric Gram, counted when "
                        "they are recorded) over the time of the WHOLE stage, which also contains the purification / Newton-Schulz "
                        "rounds and the Cholesky kernels (their flops are not counted: a lower bound).  Replicated on every rank; "
                        "~43 dependency levels and ~85 purification rounds per step, each a grid barrier + one wave of 32 x 32 DMMA "
                        "tiles: the stage is latency-bound, the GEMM units run at 18-19 TFLOP/s inside their k-loops (L2 operand "
                        "bandwidth 31.5 B/clk/SM = the DMMA rate for 32 x 32 tiles; plain DFMA 2.9 TFLOP/s)"})
    # (a) query contraction
    flops_a = 8.0 * BATCH * r0 * r1 * r2
    ms_a = st.get("query_fwd", 0.0) + st.get("query_bwd", 0.0)
    ach_a = flops_a / (ms_a * 1e-3) / 1e12 if ms_a > 0 else None
    out.append({"family": "a: query contraction core x1 r x2 s, forward + backward", "bound": "fp32-ffma", "achieved": ach_a,
                "peak": FFMA_PEAK_TF, "unit": "TFLOP/s", "frac": ach_a / FFMA_PEAK_TF if ach_a else None,
                "peak_source": "nominal FP32 FFMA", "algorithmic_flops_per_step": flops_a, "ms_per_step": ms_a,
                "share_of_step": share(["query_fwd", "query_bwd"])})
    # (d) fused filtered evaluation
    if eval_ms:
        flops_d = 2.0 * BATCH * n_local * r2
        ach_d = flops_d / (eval_ms * 1e-3) / 1e12
        tc_eval = r2 >= 64 and n_local >= 1024          # rt_score_rank_fused takes the tensor-core path for these shapes
        peak_d = tf_burst / 6.0 if tc_eval else FFMA_PEAK_TF
        out.append({"family": "d: fused score + filtered rank (evaluation batch of 512)",
                    "bound": "tensor" if tc_eval else "fp32-ffma",
                    "achieved": ach_d, "peak": peak_d, "unit": "TFLOP/s", "frac": ach_d / peak_d,
                    "peak_source": (src + " bf16_tflops / 6 (fp32-accurate logits = 3 TF32 MMAs at half the bf16 rate; exact fp32 "
                                    "re-check of the band around the target)") if tc_eval
                                   else "nominal FP32 FFMA (ranks need fp32-accurate scores)",
                    "algorithmic_flops_per_batch": flops_d,
                    "ms_per_batch": eval_ms, "share_of_step": None})
    return out


_T0 = time.time()


def progress(msg):
    """Phase marker on stderr (RT_BENCH_LOG=1): where a multi-GPU run is when it stops answering."""
    if os.environ.get("RT_BENCH_LOG", "0") == "1":
        print(f"[bench +{time.time() - _T0:6.1f}s rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="wn18rr", choices=list(WORKLOADS))
    ap.add_argument("--variant", type=int, default=3,
                    help="fused score kernel: 3 = tcgen05 3xTF32 at fp32 accuracy (1e-5 parity, the default), 0 = fp32 FFMA "
                         "(1e-5 parity), 1 = tcgen05 TF32 (2e-3), 2 = warp-specialised tcgen05 with scaled fp16 operands "
                         "(2e-3; does not train from the reference's initialisation, profiles/r02_train_wn18rr_head_v*.json)")
    ap.add_argument("--cpu-steps", type=int, default=6, help="reference steps timed for cpu_baseline (0 = skip)")
    ap.add_argument("--torch-gpu-steps", type=int, default=4, help="reference-port steps on CUDA tensors (0 = skip)")
    ap.add_argument("--eval-batches", type=int, default=8)
    ap.add_argument("--no-graphs", action="store_true", help="launch kernels eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-large-kernel", action="store_true", help="skip timing the fused kernel on the 1M-entity shard")
    ap.add_argument("--no-strict", action="store_true", help="skip the run with the other score kernel (variant 2 <-> 0)")
    ap.add_argument("--no-c5", action="store_true", help="skip the synthetic 1M-entity sub-record")
    ap.add_argument("--c5-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (loss, ||rgrad||, core, relation factor, "
                         "a seeded sample of entity-factor rows) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the CUDA path's results: it needs --impl b200")
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: rtucker_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the communicator is created; rank 0 must print ONE JSON line,
        # so stdout points at stderr until the communicator exists
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            group = dist.group.WORLD
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    from rtucker_b200 import lib

    w, graph, data_label = load_workload(args.workload)
    use_graphs = not args.no_graphs and (world == 1 or os.environ.get("RT_GRAPH_NCCL", "1") == "1")
    total_steps = args.warmup + args.steps
    run = Runner(w, graph, dev, world, rank, group, args.variant, use_graphs, 2 * total_steps)

    progress("runner built; device-resident timing")
    # ---- device-resident timing (CUDA graphs replay fit + step; inputs already in HBM) ----
    clocks = ClockSampler()
    clocks.start()
    launches0 = lib().rt_launch_count()
    ms, n_tr = run.timed_resident(args.warmup, args.steps)
    launches_eager = int(lib().rt_launch_count() - launches0)
    value = n_tr / (ms * 1e-3)
    eng = run.opt._engine
    if args.dump_outputs:                    # before the profile and e2e passes below take further steps
        run.dump_outputs(args.dump_outputs)

    progress(f"resident done: {ms / args.steps:.3f} ms/step; stage profile")
    # ---- per-stage profile pass: same steps launched eagerly with CUDA-event brackets around every stage
    #      (the graph path cannot be bracketed); also counts the kernels of one step ----
    prof_steps = min(args.steps, 10)
    for i in range(2):                       # two untimed eager steps: the first eager launches after graph replay stall
        run.one_step(*run.dev_batches[i])
    eng.timers = {}
    l0 = lib().rt_launch_count()
    f0 = lib().rt_small_flop_count()
    run.barrier()
    for i in range(prof_steps):
        run.one_step(*run.dev_batches[args.warmup + i])
    run.barrier()
    launches_per_step = int(lib().rt_launch_count() - l0) // prof_steps
    small_flops_per_step = float(lib().rt_small_flop_count() - f0) / prof_steps
    stage_ms = eng.stage_ms()
    eng.timers = None
    launches = launches_per_step * args.steps if launches_eager <= 2 * args.steps else launches_eager

    progress("stage profile done; e2e")
    # ---- end to end: host batches in, loss out, every step ----
    ms_e2e, tr_e2e, h2d, d2h = run.timed_e2e(total_steps, args.steps)
    clock_info = clocks.stop()
    e2e_value = tr_e2e / (ms_e2e * 1e-3)

    progress("e2e done; eval")
    # ---- filtered evaluation ----
    eval_qps = eval_ms = None
    if args.eval_batches > 0:
        eval_qps, eval_ms = run.eval_qps(args.eval_batches, w.get("eval"))

    progress("eval done; score kernel timing")
    score_timing = time_score_kernel(run, dev, args.variant, args.steps,
                                     large=(world == 1 and args.workload != "synthetic-1m" and not args.no_large_kernel))

    progress("score timing done; other variant")
    # ---- the other score kernel on the same batches ----
    strict = fast = None
    if not args.no_strict:
        other = 0 if args.variant != 0 else 3
        del run.dev_batches
        run0 = Runner(w, graph, dev, world, rank, group, other, use_graphs, total_steps)
        ms0, tr0 = run0.timed_resident(args.warmup, args.steps)
        rec = {"value": tr0 / (ms0 * 1e-3), "ms_per_step": ms0 / args.steps}
        if other == 0:
            strict = dict(rec, note="score kernel variant 0 (fp32 FFMA, 1e-5 parity path), everything else identical")
        elif other == 3:
            fast = dict(rec, note="score kernel variant 3 (3xTF32 tensor-core path at fp32 accuracy), everything else identical")
        else:
            fast = dict(rec, note="score kernel variant 2 (fp16-operand tcgen05, 2e-3 kernel tolerance), everything else identical. "
                                  "NOT the headline: on real WN18RR from the reference's initialisation it does not learn (valid MRR "
                                  "stays at chance while variant 0 reaches 0.067 in 30 epochs, profiles/r02_train_wn18rr_head_v*.json): "
                                  "the 11-bit rounding of the entity factor leaks the large in-span part of dL/dO into the tangent space")
        del run0
        torch.cuda.empty_cache()

    progress("other variant done; c5")
    # ---- BASELINE configs[4]: synthetic 1M entities, rank (200,200,200), on the same ranks ----
    c5 = None
    if not args.no_c5 and args.workload != "synthetic-1m":
        try:
            w5 = dict(WORKLOADS["synthetic-1m"])
            g5 = synth_graph(w5)
            n5 = 3 + args.c5_steps
            run5 = Runner(w5, g5, dev, world, rank, group, args.variant, False, n5)
            ms5, tr5 = run5.timed_resident(3, args.c5_steps)
            q5, _ = run5.eval_qps(2)
            c5 = {"workload": "synthetic-1m: N=1,000,000 entities, M=1000 relations, rank (200,200,200), batch 512, rsgd",
                  "value": tr5 / (ms5 * 1e-3), "unit": "triples/s", "ms_per_step": ms5 / args.c5_steps, "steps": args.c5_steps,
                  "warmup": 3, "eval_queries_per_s": q5, "n_gpus": world, "cuda_graphs": False}
            del run5
            torch.cuda.empty_cache()
        except RuntimeError as exc:
            c5 = {"error": str(exc)[:200]}

    progress("c5 done; teardown")
    if world > 1:
        # No destroy_process_group(): with CUDA graphs that captured NCCL kernels still alive it never returned (measured:
        # both ranks reached this line after 25 s and sat in the destructor until the driver's limit).  Every rank
        # synchronises, passes one last barrier and leaves through os._exit once its output is flushed.
        torch.cuda.synchronize()
        torch.distributed.barrier()
        torch.cuda.synchronize()
    if rank != 0:
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peaks = json.load(open(peaks_path)) if os.path.isfile(peaks_path) else {}
    n_local = run.n_end - run.n_begin
    roof_all = rooflines(w, n_local, ms / args.steps, stage_ms, score_timing, eval_ms, peaks, small_flops_per_step)
    measurable = [r for r in roof_all if r.get("frac") is not None and r.get("share_of_step") is not None]
    dominant = max(measurable, key=lambda r: r["share_of_step"]) if measurable else roof_all[0]
    roofline = {k: dominant.get(k) for k in ("bound", "achieved", "peak", "unit", "frac", "traffic")}
    roofline.update({"kernel": dominant["family"], "share_of_step": dominant["share_of_step"],
                     "peak_source": dominant.get("peak_source"),
                     "note": "the measurable kernel family with the largest share of the step; every family is in roofline_all"})

    cpu = gpu_torch = None
    if world == 1:
        if args.cpu_steps > 0:
            tps, sps, cores = reference_steps(w, graph, args.cpu_steps, 1, threads=os.cpu_count())
            cpu = {"value": tps, "unit": "triples/s", "cores": cores, "kind": "port",
                   "sample": f"{args.cpu_steps} full train steps of B={BATCH} after 1 warm-up (oracle/reference_step.py: "
                             f"the reference's autodiff-through-rank-2r step), {sps:.3f} s/step; dense targets built outside the timed region"}
        if args.torch_gpu_steps > 0:
            try:
                tps, sps, _ = reference_steps(w, graph, args.torch_gpu_steps, 2, device="cuda")
                gpu_torch = {"value": tps, "unit": "triples/s", "ms_per_step": sps * 1e3, "kind": "port on CUDA tensors",
                             "sample": f"{args.torch_gpu_steps} steps after 2 warm-ups of the same reference-step port with every tensor "
                                       "on this GPU (stock cuBLAS / cuSOLVER / ATen, dense 512 x N targets resident on the device)"}
            except RuntimeError as exc:
                gpu_torch = {"error": str(exc)[:200]}

    line = {
        "metric": metric_name(data_label), "value": value, "unit": "triples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 (score GEMMs: f16 operands / f32 accumulate; N x r x r passes 3xTF32; N-independent stage f64)" if args.variant == 2 else
                 ("f32 (score GEMMs tf32)" if args.variant == 1 else
                  ("f32 (score GEMMs and N x r x r passes: 3xTF32 on tcgen05 with round-to-nearest partial sums = fp32 accuracy, "
                   "1e-5 parity; Grams and N-independent stage f64)" if args.variant == 3 else
                   "f32 (score GEMMs fp32 FFMA; N x r x r passes 3xTF32 with round-to-nearest partial sums = fp32 accuracy; Grams and N-independent stage f64)")),
        "data": data_label,
        "config": dict(config_dict(w, args), note="entity-sharded over %d GPU(s)" % world),
        "queries_per_s": BATCH * args.steps / (ms * 1e-3),
        "eval_queries_per_s": eval_qps,
        "eval_note": "filtered ranking of the real test split (first batches)" if w.get("eval") is not None else "train queries re-ranked",
        "value_strict_fp32": strict,
        "value_variant2": fast,
        "e2e": {"value": e2e_value, "unit": "triples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches,
        "gpu_launches_note": "kernels of this library executed in the timed region (%d per step; replayed from 2 CUDA graphs per step when graphs are on)" % launches_per_step,
        "cuda_graphs": bool(eng.use_graphs and eng._graphs),
        "roofline": roofline,
        "roofline_all": roof_all,
        "stage_ms": stage_ms,
        "stage_ms_note": "median ms per stage over %d EAGERLY launched steps (CUDA events on the launching stream): stages made "
                         "of several launches include host launch gaps, so the sum exceeds ms_per_step, which is "
                         "measured on the CUDA-graph path; shares in roofline_all are shares of this sum" % prof_steps,
        "cpu_baseline": cpu,
        "torch_gpu_baseline": gpu_torch,
        "c5": c5,
        "clocks": clock_info,
    }
    print(json.dumps(line))
    if world > 1:          # see the teardown note above: leave without running the communicator's destructor
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
