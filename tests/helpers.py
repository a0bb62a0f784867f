"""Shared helpers for the parity tests (GPU box and build container)."""
import json
import os

import numpy as np
import torch

from oracle import torch_port as tp

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL, ATOL = 1e-3, 1e-4          # BASELINE.json north_star: fp32 parity tolerance


def cases(kind):
    with open(os.path.join(GOLDEN, "cases.json")) as f:
        return json.load(f)[kind]


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def case_params(c, device=None):
    p = tp.synthetic_params(c["N"], c["W"], c["H"], c["multi"], seed=c["pseed"], scale_mode=c["mode"])
    if device is not None:
        p = {k: v.to(device) for k, v in p.items()}
    return p


def build_model(c, device, params=None):
    """The drop-in Model loaded with the case's seeded weights."""
    from models.base_model import Model
    m = Model(c["N"], 2, c["W"], c["multi"], horizon=c["H"])
    m.load_state_dict(params if params is not None else case_params(c))
    return m.to(device)


def reference_default_init(N, W, H, multi, g):
    """The reference Model's own default init (torch.manual_seed(0) before construction, main.py:52) as a state_dict.
    The drop-in Model creates the same tensors in the same order, so it draws them; the per-tensor sums the reference's
    init left in golden `g` (oracle/make_golden.py) confirm that they are the reference's."""
    from models.base_model import Model
    torch.manual_seed(0)
    sd = {k: v.detach().clone() for k, v in Model(N, 2, W, multi, horizon=H).state_dict().items()}
    assert sorted("init_sum." + k for k in sd) == sorted(f for f in g.files if f.startswith("init_sum."))
    for k, v in sd.items():
        a = v.double().numpy()
        np.testing.assert_allclose([a.sum(), np.abs(a).sum()], g["init_sum." + k], rtol=1e-12, atol=0, err_msg=k)
    return sd


def assert_close(actual, expected, rtol=RTOL, atol=ATOL, msg=""):
    a = actual.detach().cpu().numpy() if torch.is_tensor(actual) else np.asarray(actual)
    e = expected.detach().cpu().numpy() if torch.is_tensor(expected) else np.asarray(expected)
    assert a.shape == e.shape, f"{msg}: shape {a.shape} vs {e.shape}"
    err = np.abs(a.astype(np.float64) - e.astype(np.float64))
    tol = atol + rtol * np.abs(e.astype(np.float64))
    bad = err > tol
    if bad.any():
        i = np.unravel_index(np.argmax(err - tol), err.shape)
        raise AssertionError(f"{msg}: {bad.sum()}/{bad.size} elements outside rtol={rtol} atol={atol}; "
                             f"worst at {i}: got {a[i]!r} want {e[i]!r} (abs err {err[i]:.3e}); "
                             f"max abs err {err.max():.3e}")
