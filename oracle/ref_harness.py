"""ORACLE / TEST INFRASTRUCTURE ONLY.

Imports the UNMODIFIED reference (a read-only checkout of R-TuckER, named by the environment
variable RTUCKER_REFERENCE_DIR) with the restated ``tucker_riemopt`` from this directory on
sys.path, and injects the module globals ``train.py`` reads implicitly (train.py:21,25,38-41,72,
183-193) -- the recipe of SURVEY.md App. E.  The reference is not part of this repository: without
it the live comparisons skip and the tests rely on the fixtures under tests/golden/ generated with it.
"""
import importlib
import os
import sys

REF_DIR = os.environ.get("RTUCKER_REFERENCE_DIR", "")
_HERE = os.path.dirname(os.path.abspath(__file__))


def available() -> bool:
    return bool(REF_DIR) and os.path.isfile(os.path.join(REF_DIR, "train.py"))


def _paths():
    os.environ.setdefault("WANDB_MODE", "disabled")
    for p in (REF_DIR, _HERE):
        if p not in sys.path:
            sys.path.insert(0, p)


def load(mode: str, opt: str = "rsgd", device: str = "cpu"):
    """Returns a namespace with the reference's train module (globals injected for
    ``mode``/``opt``), its R_TuckER and optimiser classes and the restated toolbox."""
    assert available(), "reference checkout not found"
    _paths()
    import tucker_riemopt  # restated (oracle/tucker_riemopt)
    T = importlib.import_module("train")
    sub = "symmetric" if mode == "symmetric" else "asymmetric"
    optim = importlib.import_module(f"src.model.{sub}.optim")
    model = importlib.import_module(f"src.model.{sub}.R_TuckER")
    T.MODE, T.DEVICE, T.OPT = mode, device, opt
    T.Tucker, T.SFTucker = tucker_riemopt.Tucker, tucker_riemopt.SFTucker
    T.RSGDwithMomentum, T.RGD = optim.RSGDwithMomentum, optim.RGD

    class NS:
        pass
    ns = NS()
    ns.train, ns.optim, ns.R_TuckER, ns.toolbox = T, optim, model.R_TuckER, tucker_riemopt
    ns.Data = importlib.import_module("src.data.Data").Data
    ns.KG_dataset = importlib.import_module("src.data.Dataset").KG_dataset
    ns.metrics = importlib.import_module("src.utils.metrics").metrics
    ns.filter_predictions = importlib.import_module("src.utils.utils").filter_predictions
    ns.set_random_seed = importlib.import_module("src.utils.utils").set_random_seed
    ns.Config = importlib.import_module("configs.base_config").Config
    return ns
