"""Sparse-target data pipeline (SURVEY.md section 8 row f1).

Replaces ``KG_dataset.__getitem__`` + default collate (reference src/data/Dataset.py:42-53,
train.py:226-236), which allocate a dense ``zeros(n_ent)`` row per sample (84 MB per WN18RR batch):
the (s, r) -> objects vocabulary is built once on the host as CSR, a batch is (features, CSR slice),
and only a few KB cross PCIe per step.  Item order follows the reference: train items are the unique
(s, r) pairs in first-occurrence order (Dataset.py:14-15,29-34), test items are the triples.
"""
from collections import OrderedDict

import numpy as np
import torch

from . import ops
from .engine import SparseTargets


class SparseKGDataset:
    def __init__(self, triples, n_entities, all_triples=None, test_set=False, label_smoothing=0.0):
        """triples: int array [T,3] of (s, r, o) ids for this split (reverse triples already added,
        as Data.load_data does); all_triples: every split (the filter set) when test_set."""
        triples = np.asarray(triples, dtype=np.int64).reshape(-1, 3)
        self.n_entities = int(n_entities)
        self.test_set = bool(test_set)
        self.label_smoothing = 0.0 if test_set else float(label_smoothing or 0.0)
        vocab_src = np.asarray(all_triples, dtype=np.int64).reshape(-1, 3) if test_set else triples
        vocab = OrderedDict()
        for s, r, o in vocab_src.tolist():
            vocab.setdefault((s, r), []).append(o)
        if test_set:
            self.features = triples.astype(np.int32)                      # (s, r, o) per item
            keys = [(s, r) for s, r, _ in triples.tolist()]
        else:
            pairs = OrderedDict()
            for s, r, _ in triples.tolist():
                pairs.setdefault((s, r), None)
            keys = list(pairs.keys())
            self.features = np.asarray(keys, dtype=np.int32).reshape(-1, 2)
        lists = [np.unique(np.asarray(vocab[k], dtype=np.int32)) for k in keys]  # unique + ascending
        self.counts = np.asarray([len(x) for x in lists], dtype=np.int64)
        self.off = np.zeros(len(lists) + 1, dtype=np.int64)
        np.cumsum(self.counts, out=self.off[1:])
        self.idx = np.concatenate(lists).astype(np.int32) if lists else np.zeros(0, np.int32)

    def __len__(self):
        return self.features.shape[0]

    def num_triples(self, items=None):
        """Number of (s,r,o) targets covered by ``items`` (all items if None): the 'train triples'."""
        return int(self.counts.sum() if items is None else self.counts[items].sum())

    def host_batch(self, items):
        items = np.asarray(items, dtype=np.int64)
        cnt = self.counts[items]
        off = np.zeros(len(items) + 1, dtype=np.int32)
        np.cumsum(cnt, out=off[1:])
        starts = self.off[items]
        gather = np.repeat(starts - off[:-1], cnt) + np.arange(int(off[-1]), dtype=np.int64)
        return self.features[items], off, self.idx[gather]

    def batch(self, items, device, pinned=None):
        """(features int32 [B, 2|3], SparseTargets) on ``device``; host->device copies are async from
        pinned staging buffers.  Returns also the number of bytes copied."""
        feat, off, idx = self.host_batch(items)
        tensors = []
        nbytes = 0
        for a in (feat, off, idx):
            t = torch.from_numpy(np.ascontiguousarray(a))
            if device.type == "cuda":
                t = t.pin_memory().to(device, non_blocking=True)
            nbytes += a.nbytes
            tensors.append(t)
        return tensors[0], SparseTargets(tensors[1], tensors[2]), nbytes

    def batches(self, batch_size, device, shuffle=False, drop_last=False, generator=None):
        n = len(self)
        order = torch.randperm(n, generator=generator).numpy() if shuffle else np.arange(n)
        end = n - (n % batch_size) if drop_last else n
        for lo in range(0, end, batch_size):
            items = order[lo:min(lo + batch_size, end)]
            yield (*self.batch(items, device), items)


def from_reference_data(data, split, test_set=False, label_smoothing=0.0):
    """Build a SparseKGDataset from an object with the reference ``Data`` fields
    (src/data/Data.py: entities, relations, train_data/valid_data/test_data, data)."""
    ent = {e: i for i, e in enumerate(data.entities)}
    rel = {r: i for i, r in enumerate(data.relations)}

    def ids(rows):
        return np.asarray([(ent[a], rel[b], ent[c]) for a, b, c in rows], dtype=np.int64).reshape(-1, 3)
    rows = getattr(data, f"{split}_data")
    return SparseKGDataset(ids(rows), len(data.entities), all_triples=ids(data.data) if test_set else None,
                           test_set=test_set, label_smoothing=label_smoothing)


class DeviceEpoch:
    """A split resident in HBM, iterated without host work (SURVEY.md section 8 rows f1/f2).

    Stands where the reference builds ``DataLoader(KG_dataset(...), batch_size, shuffle, drop_last, num_workers=6,
    pin_memory=True)`` (train.py:226-236): the (s, r[, o]) rows and the CSR of target lists are uploaded once
    (WN18RR train: 2.2 MB instead of 84 MB per batch), every epoch draws a permutation and each batch is assembled on
    the device by ``rt_epoch_batch``.  Iterating yields ``(features int32 [B, 2|3], SparseTargets)``.

    ``shuffle``: "device" (torch.randperm on the device: no host work at all), "host" (the reference's own draw:
    RandomSampler seeds a CPU generator from the global one and calls torch.randperm, so identical seeds give the
    reference's batches; the permutation is uploaded once per epoch), or False.
    """

    def __init__(self, dataset: SparseKGDataset, batch_size, device, shuffle="device", drop_last=False, seed=None):
        self.dataset = dataset
        self.batch_size = int(batch_size)
        self.device = torch.device(device)
        self.shuffle = shuffle
        self.drop_last = bool(drop_last)
        self.label_smoothing = dataset.label_smoothing
        self.n_entities = dataset.n_entities
        self.feat = torch.from_numpy(np.ascontiguousarray(dataset.features)).to(self.device)
        self.off = torch.from_numpy(dataset.off.astype(np.int32)).to(self.device)
        self.idx = torch.from_numpy(np.ascontiguousarray(dataset.idx)).to(self.device)
        self.counts_dev = torch.from_numpy(dataset.counts.astype(np.int64)).to(self.device)
        top = np.sort(dataset.counts)[-self.batch_size:].sum() if len(dataset) else 0
        self.cap = max(int(top), 16)            # no batch can hold more targets than the B longest lists
        self.gen = None
        if shuffle == "device":
            self.gen = torch.Generator(device=self.device)
            self.gen.manual_seed(int(seed) if seed is not None else int(torch.initial_seed()) & 0x7FFFFFFF)
        self.last_perm = None

    def __len__(self):
        n = len(self.dataset)
        return n // self.batch_size if self.drop_last else (n + self.batch_size - 1) // self.batch_size

    def num_items(self):
        n = len(self.dataset)
        return n - n % self.batch_size if self.drop_last else n

    def permutation(self):
        n = len(self.dataset)
        if self.shuffle == "device":
            return torch.randperm(n, device=self.device, generator=self.gen)
        if self.shuffle == "host":
            # torch.utils.data.RandomSampler.__iter__: seed drawn from the global generator, then randperm
            seed = int(torch.empty((), dtype=torch.int64).random_().item())
            g = torch.Generator()
            g.manual_seed(seed)
            return torch.randperm(n, generator=g).to(self.device, non_blocking=True)
        return torch.arange(n, device=self.device)

    def __iter__(self):
        perm = self.permutation()
        self.last_perm = perm
        n, B = self.num_items(), self.batch_size
        i32 = torch.int32
        fc = self.feat.shape[1]
        for lo in range(0, n, B):
            b = min(B, n - lo)
            out = (torch.empty(b, fc, dtype=i32, device=self.device), torch.empty(b + 1, dtype=i32, device=self.device),
                   torch.empty(self.cap, dtype=i32, device=self.device))
            ops.epoch_batch(perm, lo, b, self.feat, self.off, self.idx, out)
            yield out[0], SparseTargets(out[1], out[2])

    def triples_in_epoch(self):
        """Number of (s, r, o) targets the last iterated epoch covered (device tensor, no sync)."""
        perm = self.last_perm if self.last_perm is not None else torch.arange(len(self.dataset), device=self.device)
        return self.counts_dev[perm[: self.num_items()]].sum()


def wn18rr_fixture(path=None):
    """The real WN18RR triples as ids in the reference's vocabulary order (tests/golden/wn18rr_ids.npz, written by
    tests/golden/make_golden.py from the reference's Data(reverse=True)); None when the fixture is absent."""
    import os
    if path is None:
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        path = os.path.join(root, "tests", "golden", "wn18rr_ids.npz")
    if not os.path.isfile(path):
        return None
    d = np.load(path)
    # stored as column-major uint16 (every id < 65536) to keep the file small; callers get row-major int32
    split = lambda name: np.ascontiguousarray(d[name], dtype=np.int32)  # noqa: E731
    return dict(n_entities=int(d["n_entities"]), n_relations=int(d["n_relations"]),
                train=split("train"), valid=split("valid"), test=split("test"))


def datasets_from_ids(ids, label_smoothing=0.1):
    """(train, valid, test) SparseKGDataset of an id-triple dictionary (wn18rr_fixture): what train.py:226-228 builds."""
    allt = np.concatenate([ids["train"], ids["valid"], ids["test"]])
    n = ids["n_entities"]
    train = SparseKGDataset(ids["train"], n, label_smoothing=label_smoothing)
    valid = SparseKGDataset(ids["valid"], n, all_triples=allt, test_set=True)
    test = SparseKGDataset(ids["test"], n, all_triples=allt, test_set=True)
    return train, valid, test
