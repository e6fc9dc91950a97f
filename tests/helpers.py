"""Shared helpers for the parity tests: golden-fixture loading and error metrics."""
import glob
import json
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

MODEL_CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz"))
                     if not os.path.basename(p).startswith(("layers", "fit_", "dice")))


def load_case(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    case = {"cfg": json.loads(str(z["cfg"])), "X": torch.from_numpy(z["X"]), "y": torch.from_numpy(z["y"]),
            "logit": torch.from_numpy(z["logit"]), "y_pred": torch.from_numpy(z["y_pred"]),
            "loss": float(z["loss"]), "reg_loss": float(np.asarray(z["reg_loss"]).reshape(-1)[0]),
            "state": {}, "grad": {}}
    for k in z.files:
        if k.startswith("state/"):
            case["state"][k[6:]] = torch.from_numpy(z[k])
        elif k.startswith("grad/"):
            case["grad"][k[5:]] = torch.from_numpy(z[k])
    return case


def load_layers(fname="layers.npz"):
    z = np.load(os.path.join(GOLDEN_DIR, fname), allow_pickle=False)
    out = {}
    for k in z.files:
        tag, rest = k.split("/", 1)
        out.setdefault(tag, {})[rest] = torch.from_numpy(z[k])
    return out


def rel_err(a, b):
    """max|a-b| / max|b| — the parity metric of SURVEY.md §7 hard part 2."""
    a = torch.as_tensor(a).detach().to(torch.float64).reshape(-1)
    b = torch.as_tensor(b).detach().to(torch.float64).reshape(-1)
    if b.numel() == 0:
        return 0.0 if a.numel() == 0 else float("inf")
    denom = float(b.abs().max())
    if denom == 0.0:
        return float((a - b).abs().max())
    return float((a - b).abs().max()) / denom


def build_columns(cols):
    from deepctr_torch_b200.config import columns_from_cfg
    return columns_from_cfg(cols)


def build_model(cfg, device="cpu", **extra):
    """Instantiate the deepctr_torch_b200 model described by an oracle cfg dict."""
    from deepctr_torch_b200.config import model_from_cfg
    return model_from_cfg(cfg, device, **extra)


def capture_logit(model, X):
    """Run model(X) and also return the pre-sigmoid logit (recomputed from y for binary tasks is
    ill-conditioned, so hook the prediction op's inputs instead)."""
    from deepctr_torch_b200 import ops
    captured = {}
    orig = ops.predict

    def spy(terms, bias, binary=True):
        captured["logit"] = sum(t.detach().reshape(-1) for t in terms) + (bias.detach() if bias is not None else 0)
        return orig(terms, bias, binary)

    ops.predict = spy
    try:
        y = model(X)
    finally:
        ops.predict = orig
    return y, captured["logit"].reshape(-1, 1)
