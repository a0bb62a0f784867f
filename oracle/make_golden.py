"""TEST INFRASTRUCTURE — mints tests/golden/*.npz from the UNMODIFIED reference.

    STEMGNN_REFERENCE_ROOT=<microsoft/StemGNN checkout> python -m oracle.make_golden [name ...]

With names, only those files are written.  The reference `models.base_model.Model` is imported through
oracle/ref_shim.py, loaded with the seeded synthetic weights of oracle/torch_port.synthetic_params (so the
weights can be regenerated without the reference) and run on the seeded inputs of synthetic_batch.  Where
a test compares with the reference at its own default init (torch.manual_seed(0), main.py:52), the file
also holds per-tensor float64 sums of that init: the drop-in Model draws the same tensors under the same
seed, and the tests check those sums before they use its weights.  Every array written here is an output
of reference code or a data fixture (z-scored rows of the reference's dataset/ECG_data.csv); nothing of
the reference's source is stored.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_shim, torch_port  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name: (B, N, W, H, multi, param_seed, scale_mode, what)
CASES = {
    "tiny_taps":      dict(B=4, N=24, W=12, H=3, multi=5, pseed=11, mode="init", taps=True),
    "odd_h1_taps":    dict(B=3, N=37, W=12, H=1, multi=5, pseed=12, mode="trained", taps=True),
    "multi2_w8":      dict(B=5, N=19, W=8, H=2, multi=2, pseed=13, mode="trained", taps=True),
    "cfg1_shape":     dict(B=32, N=140, W=12, H=3, multi=5, pseed=14, mode="init", taps=False),
    "cfg1_trained":   dict(B=29, N=140, W=12, H=3, multi=5, pseed=15, mode="trained", taps=False),
    "cfg2_shape":     dict(B=32, N=358, W=12, H=3, multi=5, pseed=16, mode="init", taps=False),
}
GRAD_CASES = {
    "grad_multi2":    dict(B=4, N=21, W=12, H=3, multi=2, pseed=21, mode="trained", p_drop=None),
    "grad_tiny":      dict(B=4, N=24, W=12, H=3, multi=5, pseed=22, mode="trained", p_drop=None),
    "grad_dropmask":  dict(B=4, N=24, W=12, H=3, multi=2, pseed=23, mode="trained", p_drop=0.5),
}


def _ref_model(c):
    cls = ref_shim.load_reference_model_class()
    m = cls(c["N"], 2, c["W"], c["multi"], horizon=c["H"])
    p = torch_port.synthetic_params(c["N"], c["W"], c["H"], c["multi"], seed=c["pseed"],
                                    scale_mode=c["mode"])
    missing = m.load_state_dict(p, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return m, p


class _MaskDropout(torch.nn.Module):
    """stands in for model.dropout (base_model.py:103,161) with an explicit keep-mask."""
    def __init__(self, mask, p):
        super().__init__()
        self.mask, self.p = mask, p

    def forward(self, x):
        return x * self.mask / (1.0 - self.p)


def forward_case(name, c):
    m, _ = _ref_model(c)
    m.eval()
    x, _ = torch_port.synthetic_batch(c["B"], c["N"], c["W"], c["H"], seed=1234)
    out = {}
    with torch.no_grad():
        forecast, attention = m(x)
        out["forecast"] = forecast.numpy()
        if c["N"] <= 140:
            out["attention"] = attention.numpy()
        else:
            out["attention_rows7"] = attention[::7].numpy()
        if c["taps"]:
            gru_out, _ = m.GRU(x.permute(2, 0, 1).contiguous())
            out["gru_out"] = gru_out.numpy()
            mul_L, _ = m.latent_correlation_layer(x)
            out["mul_L"] = mul_L.numpy()
            X = x.unsqueeze(1).permute(0, 1, 3, 2).contiguous()
            for i in range(2):
                blk = m.stock_block[i]
                gfted = torch.matmul(mul_L.unsqueeze(1), X.unsqueeze(1))
                out[f"block{i}.iffted"] = blk.spe_seq_cell(gfted).numpy()
                fc, X = blk(X, mul_L)
                out[f"block{i}.forecast"] = fc.numpy()
                if X is not None:
                    out[f"block{i}.backcast"] = X.numpy()
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **out)
    print(name, {k: v.shape for k, v in out.items()})


def grad_case(name, c):
    m, p = _ref_model(c)
    x, y = torch_port.synthetic_batch(c["B"], c["N"], c["W"], c["H"], seed=4321)
    out = {}
    if c["p_drop"] is None:
        m.eval()
    else:
        g = torch.Generator().manual_seed(99)
        mask = (torch.rand(c["B"], c["N"], c["N"], generator=g) >= c["p_drop"]).float()
        m.dropout = _MaskDropout(mask, c["p_drop"])
        m.train()
    x.requires_grad_(True)
    forecast, attention = m(x)
    loss = torch.nn.functional.mse_loss(forecast, y)        # handler.py:140,162
    loss.backward()
    out["forecast"] = forecast.detach().numpy()
    out["attention"] = attention.detach().numpy()
    out["loss"] = np.float32(loss.item())
    out["grad.x"] = x.grad.numpy()
    for k, v in m.named_parameters():
        if v.grad is None:
            out["nograd." + k] = np.zeros(1, np.float32)
            continue
        gnp = v.grad.numpy()
        if gnp.size <= 20000:
            out["grad." + k] = gnp
        else:                                   # large GLU weights: strided sample + moments
            flat = gnp.reshape(-1)
            out["gradsample." + k] = flat[::53].copy()
            out["gradsum." + k] = np.array([flat.astype(np.float64).sum(),
                                            np.abs(flat).astype(np.float64).sum()])
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **out)
    print(name, "loss", out["loss"], len(out), "arrays")


def _init_sums(sd):
    """per-tensor float64 sum and sum of |x|: identifies a default init without storing it."""
    out = {}
    for k, v in sd.items():
        a = v.detach().double().numpy()
        out["init_sum." + k] = np.array([a.sum(), np.abs(a).sum()])
    return out


def _ref(modname):
    import importlib
    with ref_shim.reference_modules():
        return importlib.import_module(modname)


def host_logic(name):
    """tests/test_host_logic.py: the reference's metrics, dataset, rolling inference and state_dict layout."""
    from tests import test_host_logic as t
    out = {}
    ref = _ref("utils.math_utils")
    rng = np.random.default_rng(0)
    y = rng.normal(size=(17, 3, 5)); p = y + rng.normal(size=y.shape) * 0.3
    y[0, 0, 0] = 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        for j, kw in enumerate(t.METRIC_KWS):
            for i, v in enumerate(ref.evaluate(y, p, **kw)):
                out[f"metrics.{j}.{i}"] = np.asarray(v)
        out["metrics.masked_MAPE"] = np.asarray(ref.masked_MAPE(y, p))
    ref = _ref("data_loader.forecast_dataloader")
    for method in (None, "z_score", "min_max"):
        data, stat, z = t.dataset_case(method)
        ds = ref.ForecastDataset(data.copy(), 12, 3, method, dict(stat) if stat else None, interval=2)
        out[f"dataset.{method}.x_end_idx"] = np.asarray(ds.x_end_idx)
        for i in (0, 5, len(ds) - 1):
            for u, v in zip(("x", "y"), ds[i]):
                out[f"dataset.{method}.{i}.{u}"] = v.numpy()
        if method:
            out[f"dataset.{method}.de_normalized"] = ref.de_normalized(z, method, dict(stat))
    rh = _ref("models.handler")
    for emit in (1, 2, 3):
        f, tg = rh.inference(t._StubModel(emit), t._loader(), "cpu", 5, 12, 3)
        out[f"inference.{emit}.forecast"], out[f"inference.{emit}.target"] = f, tg
    out["state_dict_keys"] = np.array(list(ref_shim.build_reference_model(23, 12, 5, 3).state_dict()))
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **out)
    print(name, len(out), "arrays")


def reference_module_pickle(name):
    """handler.py:24 checkpoints pickle WHOLE modules: one written by the reference class (N=10, zeroed weights so the
    file compresses to a few kB; the loading test reads only the module structure)."""
    import pickle
    with ref_shim.reference_modules():
        import importlib
        cls = importlib.import_module("models.base_model").Model
        torch.manual_seed(0)
        m = cls(10, 2, 12, 5, horizon=3)
        with torch.no_grad():
            for v in m.parameters():
                v.zero_()
        blob = pickle.dumps(m)
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), blob=np.frombuffer(blob, np.uint8))
    print(name, len(blob), "bytes")


def default_init_n33(name):
    """tests/test_oracle_golden.py: the reference at its own default init, (B,N,W,H)=(6,33,12,3)."""
    m = ref_shim.build_reference_model(33, 12, 5, 3, seed=0).eval()
    x, _ = torch_port.synthetic_batch(6, 33, 12, 3)
    with torch.no_grad():
        f, a = m(x)
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), forecast=f.numpy(), attention=a.numpy(),
                        **_init_sums(m.state_dict()))
    print(name, f.shape, a.shape)


def cfg1_ecg(name):
    """tests/test_configs_gpu.py, BASELINE.json configs[0]: 43 consecutive z-scored ECG_data.csv rows — the 32 sliding
    windows of one batch, as the reference's loader forms them — through the reference at its default init."""
    from tests.test_configs_gpu import ecg_windows
    data = np.loadtxt(os.path.join(ref_shim.REFERENCE_ROOT, "dataset", "ECG_data.csv"), delimiter=",")
    data = (data - data.mean(0)) / data.std(0)
    rows = data[2000:2043].astype(np.float32)
    m = ref_shim.build_reference_model(140, 12, 5, 3, seed=0).eval()
    with torch.no_grad():
        f, a = m(ecg_windows(rows))
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), rows=rows, forecast=f.numpy(), attention=a.numpy(),
                        **_init_sums(m.state_dict()))
    print(name, rows.shape, f.shape)


def cfg4_reference_sample(name):
    """tests/test_configs_gpu.py, BASELINE.json configs[3] at its global batch (128,325,12,12) with the seeded weights:
    every 101st element of the reference's forecast."""
    from oracle.cpu_reference import CpuReference
    from tests.test_configs_gpu import CFG4_SAMPLE
    from tests.helpers import case_params
    c = dict(B=128, N=325, W=12, H=12, multi=5, pseed=41, mode="init")       # test_cfg4_global_batch_forward_backward
    ref = CpuReference(c["N"], c["W"], c["H"], c["multi"], case_params(c))
    assert ref.kind == "reference"
    x, _ = torch_port.synthetic_batch(c["B"], c["N"], c["W"], c["H"], seed=c["pseed"] + 1)
    f, _ = ref.forward(x)
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), forecast_sample=f.reshape(-1)[::CFG4_SAMPLE].numpy())
    print(name, f.shape)


EXTRA = {"host_logic": host_logic, "reference_module_pickle": reference_module_pickle,
         "default_init_n33": default_init_n33, "cfg1_ecg": cfg1_ecg, "cfg4_reference_sample": cfg4_reference_sample}


if __name__ == "__main__":
    assert ref_shim.reference_available(), "set STEMGNN_REFERENCE_ROOT to a microsoft/StemGNN checkout"
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    only = set(sys.argv[1:])
    for n, c in CASES.items():
        if not only or n in only:
            forward_case(n, c)
    for n, c in GRAD_CASES.items():
        if not only or n in only:
            grad_case(n, c)
    for n, fn in EXTRA.items():
        if not only or n in only:
            fn(n)
    if not only:
        import json
        with open(os.path.join(OUT, "cases.json"), "w") as f:
            json.dump({"forward": CASES, "grad": GRAD_CASES,
                       "generator": "oracle/make_golden.py", "torch": torch.__version__,
                       "reference": "microsoft/StemGNN @ dc7dea68 via oracle/ref_shim.py"}, f, indent=1)
