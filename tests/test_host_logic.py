"""CPU tests of the host-side mirror of the reference interface (handler / dataloader / metrics) and
of the C-ABI surface.  The reference's own functions were run on the same inputs by oracle/make_golden.py;
their outputs are in tests/golden/host_logic.npz."""
import os
import re

import numpy as np
import pytest
import torch

from tests.helpers import golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
METRIC_KWS = ({}, {"by_step": True}, {"by_node": True}, {"by_step": True, "by_node": True})


# ---- metrics ------------------------------------------------------------------------------------
def test_metrics_known_values():
    from utils.math_utils import MAE, MAPE, RMSE, evaluate
    y = np.array([[[1.0, 2.0], [4.0, -2.0]]])
    p = np.array([[[2.0, 2.0], [2.0, 20.0]]])
    assert MAE(y, p) == pytest.approx((1 + 0 + 2 + 22) / 4)
    assert RMSE(y, p) == pytest.approx(np.sqrt((1 + 0 + 4 + 484) / 4))
    assert MAPE(y, p) == pytest.approx((1 + 1e-5 + 1e-5 + 0.5 + 1e-5 + 5.0) / 4)   # last term clipped at 5
    m = evaluate(y, p, by_node=True)
    assert m[1].shape == (2,)
    assert evaluate(y, p, by_step=True)[2].shape == (2,)
    assert evaluate(y, p, by_step=True, by_node=True)[0].shape == (2, 2)


def test_metrics_match_reference():
    g = golden("host_logic")
    from utils import math_utils as mine
    rng = np.random.default_rng(0)
    y = rng.normal(size=(17, 3, 5)); p = y + rng.normal(size=y.shape) * 0.3
    y[0, 0, 0] = 0.0
    for j, kw in enumerate(METRIC_KWS):
        with np.errstate(divide="ignore", invalid="ignore"):
            a = mine.evaluate(y, p, **kw)
        assert len(a) == len([k for k in g.files if k.startswith(f"metrics.{j}.")])
        for i, u in enumerate(a):
            np.testing.assert_allclose(u, g[f"metrics.{j}.{i}"], rtol=1e-12)
    with np.errstate(divide="ignore", invalid="ignore"):
        np.testing.assert_allclose(mine.masked_MAPE(y, p), g["metrics.masked_MAPE"])


# ---- dataloader --------------------------------------------------------------------------------------
def test_dataset_windows_and_normalisation():
    from data_loader.forecast_dataloader import ForecastDataset, de_normalized, normalized
    data = np.arange(40, dtype=np.float64).reshape(20, 2)
    ds = ForecastDataset(data, window_size=4, horizon=2)
    assert len(ds) == 20 - 4 - 2 + 1
    x, y = ds[3]
    assert x.dtype == torch.float32 and x.shape == (4, 2) and y.shape == (2, 2)
    np.testing.assert_array_equal(x.numpy(), data[3:7]); np.testing.assert_array_equal(y.numpy(), data[7:9])
    assert len(ForecastDataset(data, 4, 2, interval=3)) == 15 // 3
    st = {"mean": data.mean(0).tolist(), "std": [0.0, data[:, 1].std()]}
    z, st2 = normalized(data, "z_score", st)
    assert st2["std"][0] == 1                                           # zero std replaced by 1
    np.testing.assert_allclose(de_normalized(z, "z_score", st2), data)
    mm, s3 = normalized(data, "min_max")
    assert mm.min() == 0.0 and mm.max() <= 1.0
    np.testing.assert_allclose(de_normalized(mm, "min_max", s3), data, atol=1e-3)


def dataset_case(method):
    """(data with NaN holes, normalisation statistics, a normalised batch to map back) for one method."""
    rng = np.random.default_rng(1)
    data = rng.normal(size=(60, 7))
    data[0, 0] = np.nan; data[10:13, 2] = np.nan; data[-1, 6] = np.nan
    stat = None
    if method == "z_score":
        stat = {"mean": np.nanmean(data, 0).tolist(), "std": np.nanstd(data, 0).tolist()}
    if method == "min_max":
        # (the reference cannot subtract the list statistics its own handler writes; use arrays)
        stat = {"min": np.nanmin(data, 0), "max": np.nanmax(data, 0)}
    return data, stat, rng.normal(size=(4, 3, 7))


@pytest.mark.parametrize("method", [None, "z_score", "min_max"])
def test_dataset_matches_reference(method):
    g = golden("host_logic")
    from data_loader import forecast_dataloader as mine
    data, stat, z = dataset_case(method)
    a = mine.ForecastDataset(data.copy(), 12, 3, method, dict(stat) if stat else None, interval=2)
    ref_idx = g[f"dataset.{method}.x_end_idx"].tolist()
    assert len(a) == len(ref_idx) and a.x_end_idx == ref_idx
    for i in (0, 5, len(a) - 1):
        for u, v in zip(a[i], ("x", "y")):
            assert torch.equal(u, torch.from_numpy(g[f"dataset.{method}.{i}.{v}"]))
    if method:
        np.testing.assert_allclose(mine.de_normalized(z, method, dict(stat)), g[f"dataset.{method}.de_normalized"])


# ---- handler: rolling inference / validate with a stub model ---------------------------------------------
class _StubModel(torch.nn.Module):
    """Emits `emit` steps per call: the mean of the window plus the step index."""
    def __init__(self, emit):
        super().__init__()
        self.emit = emit
        self.calls = 0

    def forward(self, x):
        self.calls += 1
        base = x.mean(dim=1, keepdim=True)
        out = torch.cat([base + 0.1 * (i + 1) for i in range(self.emit)], dim=1)
        return out, None


def _loader(n=23, N=5, W=12, H=3, bs=8):
    from data_loader.forecast_dataloader import ForecastDataset
    data = np.random.default_rng(2).normal(size=(n + W + H, N))
    return torch.utils.data.DataLoader(ForecastDataset(data, W, H), batch_size=bs, shuffle=False)


@pytest.mark.parametrize("emit", [3, 1, 2])
def test_inference_rolls_the_window(emit):
    from models import handler
    m = _StubModel(emit)
    loader = _loader()
    f, t = handler.inference(m, loader, "cpu", 5, 12, 3)
    assert f.shape == t.shape == (len(loader.dataset), 3, 5)
    assert m.calls == len(loader) * int(np.ceil(3 / emit))
    g = golden("host_logic")
    np.testing.assert_allclose(f, g[f"inference.{emit}.forecast"]); np.testing.assert_allclose(t, g[f"inference.{emit}.target"])


def test_validate_writes_csvs_and_scores(tmp_path, capsys):
    from models import handler
    stat = {"mean": [0.5] * 5, "std": [2.0] * 5}
    out = handler.validate(_StubModel(3), _loader(), "cpu", "z_score", stat, 5, 12, 3, result_file=str(tmp_path))
    assert set(out) == {"mae", "mae_node", "mape", "mape_node", "rmse", "rmse_node"}
    assert out["mae_node"].shape == (5,)
    for name in ("target", "predict", "predict_abs_error", "predict_ape"):
        assert (tmp_path / f"{name}.csv").exists()
    assert "RAW : MAPE" in capsys.readouterr().out


def test_save_load_roundtrip_and_epoch_naming(tmp_path):
    from models import handler
    m = torch.nn.Linear(3, 2)
    handler.save_model(m, str(tmp_path), 0)          # epoch 0 -> the "best" file name (reference quirk)
    handler.save_model(m, str(tmp_path), 4)
    assert (tmp_path / "_stemgnn.pt").exists() and (tmp_path / "4_stemgnn.pt").exists()
    m2 = handler.load_model(str(tmp_path))
    assert torch.equal(m2.weight, m.weight)
    assert handler.load_model(str(tmp_path / "nope")) is None


def test_model_state_dict_matches_reference_layout():
    """Drop-in Model: same keys/shapes as the reference state_dict (SURVEY.md §8(b)) and picklable."""
    import pickle
    from models.base_model import Model
    from oracle import torch_port as tp
    m = Model(23, 2, 12, 5, horizon=3)
    sd = m.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == tp.param_shapes(23, 12, 3)
    assert sum(p.numel() for p in m.parameters()) == 3 * 23 * 23 + 3 * 23 * 12 + 8 * 23 + 2 * 528708 + 732 + 156 + 39
    m2 = pickle.loads(pickle.dumps(m))
    assert torch.equal(m2.weight_key, m.weight_key)
    ref_keys = golden("host_logic")["state_dict_keys"].tolist()
    assert ref_keys == list(sd.keys())
    m.load_state_dict({k: torch.randn(sd[k].shape) for k in ref_keys})      # reference checkpoints load
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(2, 12, 23))
    with pytest.raises(ValueError):
        Model(23, 3, 12, 5)


# ---- C ABI surface -------------------------------------------------------------------------------------
def test_c_abi_exports_every_declared_symbol():
    from stemgnn_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "stemgnn_b200.h")).read()
    declared = set(re.findall(r"\b(stemgnn_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.stemgnn_version() == _lib.ABI_VERSION == 3
    d = _lib.Dims(32, 358, 12, 3, 5)
    import ctypes
    ev, tr = lib.stemgnn_workspace_bytes(ctypes.byref(d), 0), lib.stemgnn_workspace_bytes(ctypes.byref(d), 1)
    assert 0 < ev < tr
    bad = _lib.Dims(0, 358, 12, 3, 5)
    assert lib.stemgnn_workspace_bytes(ctypes.byref(bad), 0) == 0


def test_c_abi_rejects_bad_arguments_without_gpu():
    import ctypes
    from stemgnn_b200 import _lib
    lib = _lib.load()
    d = _lib.Dims(4, 8, 12, 3, 5)
    rc = lib.stemgnn_model_forward(ctypes.byref(d), None, None, None, None, None, None, None, 0, None)
    assert rc != 0 and b"null" in lib.stemgnn_last_error()
    with pytest.raises(RuntimeError, match="stemgnn_b200"):
        _lib.check(rc, "forward")


# ---- state_dict checkpoints (SURVEY §8(f) rank 4) ---------------------------------------------------------
def test_state_checkpoint_roundtrip_and_resume(tmp_path):
    from models import handler
    from models.base_model import Model
    from stemgnn_b200 import checkpoint as ck
    torch.manual_seed(3)
    m = Model(11, 2, 12, 2, horizon=3)
    opt = torch.optim.RMSprop(m.parameters(), lr=1e-3, eps=1e-8)
    sched = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=0.5)
    for p in m.parameters():                       # fake one optimiser step on CPU (no forward needed)
        p.grad = torch.randn_like(p) * 0.01
    opt.step(); sched.step()
    path = ck.save_checkpoint(str(tmp_path / "state.pt"), m, opt, sched, epoch=4, extra={"mae": 1.5})
    m2, c = ck.load_checkpoint(path)                                     # weights_only=True load
    assert c["epoch"] == 4 and c["extra"]["mae"] == 1.5
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k
    opt2 = torch.optim.RMSprop(m2.parameters(), lr=1e-3, eps=1e-8)
    sched2 = torch.optim.lr_scheduler.ExponentialLR(opt2, gamma=0.5)
    assert ck.restore_training(c, opt2, sched2) == 5
    assert opt2.param_groups[0]["lr"] == opt.param_groups[0]["lr"] == 5e-4
    s1, s2 = opt.state_dict()["state"], opt2.state_dict()["state"]
    assert all(torch.equal(s1[i]["square_avg"], s2[i]["square_avg"]) for i in s1)
    # reference-style whole-module pickle -> tensor-only checkpoint
    handler.save_model(m, str(tmp_path), 7)
    dst = ck.convert_module_pickle(str(tmp_path / "7_stemgnn.pt"), str(tmp_path / "conv.pt"))
    m3, _ = ck.load_checkpoint(dst)
    assert torch.equal(m3.GRU.weight_hh_l0, m.GRU.weight_hh_l0)
    with pytest.raises(RuntimeError):
        torch.save({"format": "other"}, str(tmp_path / "bad.pt"))
        ck.load_checkpoint(str(tmp_path / "bad.pt"))


def test_header_is_plain_c_and_matches_the_ctypes_layout(tmp_path):
    """include/stemgnn_b200.h compiles as C (gcc -std=c99) and its struct layout equals the ctypes mirror that
    the Python host side passes through the ABI."""
    import ctypes
    import shutil
    import subprocess
    from stemgnn_b200 import _lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "abi.c"
    src.write_text('''
#include <stdio.h>
#include <stddef.h>
#include "stemgnn_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu\\n", sizeof(stemgnn_dims_t), sizeof(stemgnn_block_params_t), sizeof(stemgnn_params_t),
         sizeof(stemgnn_fwd_opts_t), sizeof(stemgnn_grads_t));
  printf("%zu %zu %zu %zu\\n", offsetof(stemgnn_params_t, block), offsetof(stemgnn_params_t, fc0_w),
         offsetof(stemgnn_block_params_t, glu_left_w), offsetof(stemgnn_block_params_t, glu_right_b));
  printf("%zu %zu %zu %zu\\n", offsetof(stemgnn_fwd_opts_t, dropout_seed), offsetof(stemgnn_fwd_opts_t, dropout_mask),
         offsetof(stemgnn_fwd_opts_t, gemm_mode), offsetof(stemgnn_fwd_opts_t, reuse_folded));
  return 0;
}
''')
    exe = tmp_path / "abi"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    sizes = [int(v) for v in out]
    assert sizes[:5] == [ctypes.sizeof(_lib.Dims), ctypes.sizeof(_lib.BlockPtrs), ctypes.sizeof(_lib.ModelPtrs),
                         ctypes.sizeof(_lib.FwdOpts), ctypes.sizeof(_lib.ModelPtrs)]
    assert sizes[5:9] == [_lib.ModelPtrs.block.offset, _lib.ModelPtrs.fc0_w.offset,
                          _lib.BlockPtrs.glu_left_w.offset, _lib.BlockPtrs.glu_right_b.offset]
    assert sizes[9:13] == [_lib.FwdOpts.dropout_seed.offset, _lib.FwdOpts.dropout_mask.offset,
                           _lib.FwdOpts.gemm_mode.offset, _lib.FwdOpts.reuse_folded.offset]


def test_reference_made_module_pickle_loads_into_dropin(tmp_path):
    """handler.py:24 saves WHOLE modules: a checkpoint written by the reference class must unpickle into the
    drop-in class of the same module path and be usable (ADVICE r1: __setstate__ fills what the reference lacks)."""
    import pickle
    import models.base_model as ours
    blob = golden("reference_module_pickle")["blob"].tobytes()     # pickled by the reference class (N=10)
    m = pickle.loads(blob)
    assert type(m) is ours.Model and type(m.stock_block[1]) is ours.StockBlockLayer
    assert m._rt is None and m.gemm_mode == 0 and m.dropout_rate == 0.5 and m.multi_layer == 5
    assert m.stock_block[0].gemm_mode == 0
    with pytest.raises(RuntimeError, match="CUDA"):          # reaches the runtime, which refuses CPU tensors
        m(torch.zeros(2, 12, 10))


def test_runtime_cache_follows_replaced_parameters():
    """ADVICE r1: the cached raw-pointer struct is rebuilt when a Parameter object or its storage is replaced."""
    from models.base_model import Model
    import torch.nn as nn
    m = Model(6, 2, 12, 5, horizon=3)
    seen = []
    import stemgnn_b200.runtime as rt
    orig = rt.build_ptrs
    try:
        rt.build_ptrs = lambda tensors: seen.append(tensors["weight_key"].data_ptr()) or object()
        r1 = m._runtime()
        assert m._runtime() is r1 and len(seen) == 1                      # cached while nothing changes
        m.weight_key = nn.Parameter(torch.ones(6, 1))
        r2 = m._runtime()
        assert r2 is not r1 and seen[-1] == m.weight_key.data_ptr()
        m.weight_query.data = torch.zeros(6, 1)
        assert m._runtime() is not r2
    finally:
        rt.build_ptrs = orig


def test_interleaved_chebyshev_rows_make_gfted_rows_dense():
    """The layout identity behind the coalesced graph-Fourier epilogue (csrc/spec_tc.cu): with the A-operand rows ordered
    m' = node*3 + k', the chain's input G[(b*N + node)*3W + k'*W + t] is the dense array G[b][m'][t] of shape (B, 3N, W), and
    the copy kernel's permutation (stack_n = N, row_mul = 3) produces exactly that row order from the stacked mul_L[1..3]."""
    B, N, W = 3, 7, 4
    for b in range(B):
        for node in range(N):
            for kp in range(3):
                for t in range(W):
                    assert (b * N + node) * 3 * W + kp * W + t == (b * 3 * N + node * 3 + kp) * W + t
    rows = 3 * N
    dst = {}
    for r in range(rows):                      # pad_rows_kernel, stack_n > 0: r = k*stack_n + i -> i*row_mul + k + row_add
        dst[(r % N) * 3 + r // N] = r
    assert sorted(dst) == list(range(rows))
    for node in range(N):
        for kp in range(3):
            assert dst[node * 3 + kp] == kp * N + node       # row node*3 + k' holds mul_L[k'+1][node][:]
