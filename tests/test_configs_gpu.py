"""BASELINE.json configs on the B200 (VERDICT r1 "N3"): every named configuration runs through the CUDA path and
is compared with the reference — its stored outputs (tests/golden/, oracle/make_golden.py) and the torch port of it.

  cfg1  ECG_data.csv N=140 W=12 H=3 batch=32: forward on real ECG rows vs the reference at its default init;
  cfg3  (64,228,12,3) bf16 tensor-core mode with its own, looser, stated tolerance;
  cfg4  global batch (128,325,12,12): forward + backward;
  cfg5  N=2048 (>= 8 windows): forward + backward.
"""
import numpy as np
import pytest
import torch

from oracle import torch_port as tp
from tests.helpers import assert_close, build_model, case_params, golden, reference_default_init

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CFG4_SAMPLE = 101          # tests/golden/cfg4_reference_sample.npz holds every 101st forecast element


def ecg_windows(rows, B=32, W=12):
    """(B, W, N): the B sliding windows over consecutive rows (ForecastDataset with interval=1, shuffle=False)."""
    return torch.from_numpy(np.stack([rows[i:i + W] for i in range(B)]))


def test_cfg1_ecg_forward_vs_live_reference():
    """configs[0]: z-scored ECG rows, reference default-seed weights, CUDA forward vs the unmodified reference."""
    g = golden("cfg1_ecg")
    x = ecg_windows(g["rows"])
    sd = reference_default_init(140, 12, 3, 5, g)
    from models.base_model import Model
    m = Model(140, 2, 12, 5, horizon=3)
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval()
    with torch.no_grad():
        f, a = m(x.to(DEV))
    f_ref = torch.from_numpy(g["forecast"])
    assert_close(f, f_ref, msg="cfg1 forecast vs live reference")
    assert_close(a, g["attention"], msg="cfg1 attention vs live reference")
    mae = float((f.cpu() - f_ref).abs().mean())
    assert mae < 2e-5, mae


def _fwd_bwd_vs_cpu(B, N, H, seed, rtol_g, reference_sample=None):
    c = dict(B=B, N=N, W=12, H=H, multi=5, pseed=seed, mode="init")
    p = case_params(c)
    x, y = tp.synthetic_batch(B, N, 12, H, seed=seed + 1)
    m = build_model(c, DEV, p)
    m.eval()                                           # eval: no dropout, gradients still flow
    f, a = m(x.to(DEV))
    loss = torch.nn.functional.mse_loss(f, y.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    pr = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    f_ref, a_ref = tp.model_forward(x, pr)
    torch.nn.functional.mse_loss(f_ref, y).backward()
    if reference_sample is not None:           # the port itself is re-checked against the reference's stored forecast
        assert_close(f_ref.detach().reshape(-1)[::CFG4_SAMPLE], golden(reference_sample)["forecast_sample"],
                     rtol=1e-4, atol=1e-5, msg="port vs live reference")
    assert_close(f.detach(), f_ref.detach(), msg="forecast")
    assert_close(a.detach(), a_ref.detach(), msg="attention")
    named = dict(m.named_parameters())
    worst = 0.0
    for k, g_ref in ((k, v.grad) for k, v in pr.items()):
        g = named[k].grad
        if g_ref is None or float(g_ref.abs().max()) == 0.0:
            continue
        assert g is not None, k
        rel = float((g.cpu() - g_ref).abs().max() / g_ref.abs().max())
        worst = max(worst, rel)
        assert rel < rtol_g, f"{k}: gradient rel err {rel:.3e}"
    return worst


def test_cfg4_global_batch_forward_backward():
    """configs[3] at its global batch on one GPU: (128,325,12,12)."""
    _fwd_bwd_vs_cpu(128, 325, 12, 41, 1e-2, "cfg4_reference_sample")    # default mode: weight / input gradient GEMMs on TF32 tensor cores


def test_cfg5_n2048_forward_backward():
    """configs[4] node count: (8,2048,12,3) — the GRU runs beyond the single-cluster envelope."""
    _fwd_bwd_vs_cpu(8, 2048, 3, 43, 1e-2)


def test_cfg3_bf16_mode():
    """configs[2] "bf16 tensor-core GFT": (64,228,12,3) with Model.gemm_mode = GEMM_BF16.
    Stated tolerance for this mode: rtol 1e-2 / atol 2e-3 on the forecast (bf16 operands carry 8 mantissa bits;
    SURVEY §7.3 measured 7.7e-2 stage-level error for a bf16 GFT, which the heads attenuate), attention exact-path."""
    from stemgnn_b200 import runtime
    if not hasattr(runtime, "GEMM_BF16"):
        pytest.skip("bf16 mode not built")
    c = dict(B=64, N=228, W=12, H=3, multi=5, pseed=328, mode="trained")
    p = case_params(c)
    m = build_model(c, DEV, p).eval()
    m.gemm_mode = runtime.GEMM_BF16
    x, _ = tp.synthetic_batch(64, 228, 12, 3, seed=99)
    with torch.no_grad():
        f_ref, a_ref = tp.model_forward(x, p)
        f, a = m(x.to(DEV))
    assert_close(a, a_ref, msg="attention (GRU/attention stay in split-precision fp32)")
    assert_close(f, f_ref, rtol=1e-2, atol=2e-3, msg="bf16 forecast")
