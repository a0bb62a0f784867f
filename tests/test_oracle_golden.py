"""The oracle (oracle/stemgnn_oracle.py numpy restatement and oracle/torch_port.py) is pinned
against golden vectors produced by the UNMODIFIED reference (oracle/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import stemgnn_oracle as so, torch_port as tp
from tests.helpers import reference_default_init

RTOL, ATOL = 1e-3, 1e-4        # BASELINE.json north_star tolerance (fp32)
TIGHT = dict(rtol=2e-4, atol=2e-5)


def _cases(golden_dir, kind):
    with open(os.path.join(golden_dir, "cases.json")) as f:
        return json.load(f)[kind]


def _params_np(c):
    p = tp.synthetic_params(c["N"], c["W"], c["H"], c["multi"], seed=c["pseed"], scale_mode=c["mode"])
    return p, {k: v.numpy() for k, v in p.items()}


@pytest.mark.parametrize("name", ["tiny_taps", "odd_h1_taps", "multi2_w8", "cfg1_shape",
                                  "cfg1_trained"])
def test_numpy_oracle_matches_reference_golden(golden_dir, name):
    c = _cases(golden_dir, "forward")[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    _, p = _params_np(c)
    x, _ = tp.synthetic_batch(c["B"], c["N"], c["W"], c["H"], seed=1234)
    taps = {}
    forecast, attention = so.model_forward(x.numpy(), p, taps=taps)
    np.testing.assert_allclose(forecast, g["forecast"], **TIGHT)
    np.testing.assert_allclose(attention, g["attention"], **TIGHT)
    if c["taps"]:
        np.testing.assert_allclose(taps["gru_out"], g["gru_out"], **TIGHT)
        np.testing.assert_allclose(taps["mul_L"], g["mul_L"], **TIGHT)
        for i in range(2):
            np.testing.assert_allclose(taps[f"block{i}.iffted"], g[f"block{i}.iffted"], **TIGHT)
            np.testing.assert_allclose(taps[f"block{i}.forecast"], g[f"block{i}.forecast"], **TIGHT)


@pytest.mark.parametrize("name", ["tiny_taps", "odd_h1_taps", "multi2_w8", "cfg1_shape",
                                  "cfg1_trained", "cfg2_shape"])
def test_torch_port_matches_reference_golden(golden_dir, name):
    c = _cases(golden_dir, "forward")[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    p, _ = _params_np(c)
    x, _ = tp.synthetic_batch(c["B"], c["N"], c["W"], c["H"], seed=1234)
    with torch.no_grad():
        forecast, attention = tp.model_forward(x, p)
    np.testing.assert_allclose(forecast.numpy(), g["forecast"], **TIGHT)
    if "attention" in g:
        np.testing.assert_allclose(attention.numpy(), g["attention"], **TIGHT)
    else:
        np.testing.assert_allclose(attention.numpy()[::7], g["attention_rows7"], **TIGHT)


@pytest.mark.parametrize("name", ["grad_multi2", "grad_tiny", "grad_dropmask"])
def test_torch_port_gradients_match_reference_golden(golden_dir, name):
    c = _cases(golden_dir, "grad")[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    p, _ = _params_np(c)
    for v in p.values():
        v.requires_grad_(True)
    x, y = tp.synthetic_batch(c["B"], c["N"], c["W"], c["H"], seed=4321)
    x.requires_grad_(True)
    mask = None
    if c["p_drop"] is not None:
        gen = torch.Generator().manual_seed(99)
        mask = (torch.rand(c["B"], c["N"], c["N"], generator=gen) >= c["p_drop"]).float()
    forecast, _ = tp.model_forward(x, p, dropout_mask=mask, dropout_p=c["p_drop"] or 0.5)
    loss = torch.nn.functional.mse_loss(forecast, y)
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) < 1e-5
    np.testing.assert_allclose(x.grad.numpy(), g["grad.x"], rtol=1e-3, atol=1e-6)
    for k in g.files:
        if k.startswith("grad.") and k != "grad.x":
            np.testing.assert_allclose(p[k[5:]].grad.numpy(), g[k], rtol=1e-3, atol=1e-6, err_msg=k)
        elif k.startswith("gradsample."):
            np.testing.assert_allclose(p[k[11:]].grad.numpy().reshape(-1)[::53], g[k],
                                       rtol=1e-3, atol=1e-6, err_msg=k)
        elif k.startswith("nograd."):
            assert p[k[7:]].grad is None or float(p[k[7:]].grad.abs().max()) == 0.0


def test_param_shapes_and_count():
    assert so.parameter_count(358, 12, 3) == 1458587      # SURVEY.md §8(a) a1 [measured]
    assert so.parameter_count(140, 12, 3) == 1123303
    shapes = tp.param_shapes(140, 12, 3)
    assert sum(int(np.prod(s)) for s in shapes.values()) == 1123303
    assert abs(so.forward_flops(32, 358, 12, 3) / 1e9 - 28.3) < 0.2   # SURVEY.md §8(d)


def test_oracle_against_live_reference_default_init(golden_dir):
    """Reference Model at its OWN default init (torch.manual_seed(0), main.py:52) vs both restatements —
    independent of the synthetic weights."""
    g = np.load(os.path.join(golden_dir, "default_init_n33.npz"))
    sd = reference_default_init(33, 12, 3, 5, g)
    assert {k: tuple(v.shape) for k, v in sd.items()} == tp.param_shapes(33, 12, 3)
    x, _ = tp.synthetic_batch(6, 33, 12, 3)
    f_ref, a_ref = g["forecast"], g["attention"]
    with torch.no_grad():
        f_port, a_port = tp.model_forward(x, sd)
    f_np, a_np = so.model_forward(x.numpy(), {k: v.numpy() for k, v in sd.items()})
    np.testing.assert_allclose(f_port.numpy(), f_ref, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(a_port.numpy(), a_ref, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(f_np, f_ref, **TIGHT)
    np.testing.assert_allclose(a_np, a_ref, **TIGHT)
