"""Helpers shared by the CPU and GPU tests to read tests/golden/*.npz."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=True)


def step_fixture(name):
    z = load(name)
    sym = "init_E" in z.files
    init = {k[5:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("init_")}
    batches = []
    for i in range(z["sub"].shape[0]):
        batches.append((torch.from_numpy(z["rel"][i]), torch.from_numpy(z["sub"][i]),
                        torch.from_numpy(z["off"][i]), torch.from_numpy(np.asarray(z["idx"][i], dtype=np.int64))))
    # the final dense tensor, stored as its exact Tucker factors (make_golden.tucker_factors)
    X_final = np.einsum("ijk,ai,bj,ck->abc", z["X_final_core"], z["X_final_U0"], z["X_final_U1"], z["X_final_U2"])
    return dict(sym=sym, init=init, batches=batches, loss=z["loss"], norm=z["norm"], X_final=torch.from_numpy(X_final),
                ls=float(z["ls"]), reg=float(z["reg"]), lr=float(z["lr"]), beta=float(z["beta"]),
                rank=tuple(int(x) for x in z["rank"]), N=int(z["N"]), M=int(z["M"]))
