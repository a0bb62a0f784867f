"""TEST INFRASTRUCTURE — not product code.

Loads the UNMODIFIED reference (microsoft/StemGNN) from the checkout named by the environment variable
STEMGNN_REFERENCE_ROOT.  `oracle/make_golden.py` mints `tests/golden/` from it; `bench.py --impl reference`
and `cpu_baseline` use it when it is set and the torch port otherwise.  The tests never need it: what they
compare against the reference is stored under `tests/golden/`.

The reference pins torch==1.7.1 (requirements.txt:4) and uses four APIs that no longer
exist on the container stack (torch 2.11 / numpy 2.3 / pandas 3.0).  They are patched
*around* the reference (no reference file is edited or copied):

  1. torch.rfft(x, 1, onesided=False)        (models/base_model.py:49)
       -> view_as_real(torch.fft.fft(x, dim=-1))
  2. torch.irfft(X, 1, onesided=False)       (models/base_model.py:58)
       -> torch.fft.irfft(view_as_complex(X), n=X.shape[-2], dim=-1)
     torch 1.7's C2R back-ends (MKL conjugate-even storage, cuFFT C2R) consume only bins
     0..n/2 and ignore Im(DC) / Im(Nyquist); that is what torch.fft.irfft does too.  This is
     the one residual risk of the pin (torch 1.7.1 itself cannot be installed here).
  3. np.float                                 (models/handler.py:50)
  4. DataFrame.fillna(method=...)             (data_loader/forecast_dataloader.py:49)
     torch.load(weights_only default)         (models/handler.py:37)
"""
import contextlib
import importlib
import os
import sys

REFERENCE_ROOT = os.environ.get("STEMGNN_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "models", "base_model.py"))


def _install_patches():
    import numpy as np
    import torch

    if not hasattr(torch, "_stemgnn_shim"):
        def _rfft(x, signal_ndim, normalized=False, onesided=True):
            assert signal_ndim == 1 and not normalized and not onesided
            return torch.view_as_real(torch.fft.fft(x, dim=-1))

        def _irfft(x, signal_ndim, normalized=False, onesided=True, signal_sizes=None):
            assert signal_ndim == 1 and not normalized and not onesided
            n = x.shape[-2]
            return torch.fft.irfft(torch.view_as_complex(x.contiguous()), n=n, dim=-1)

        torch.rfft = _rfft
        torch.irfft = _irfft
        _orig_load = torch.load

        def _load(*a, **kw):
            kw.setdefault("weights_only", False)
            return _orig_load(*a, **kw)

        torch.load = _load
        torch._stemgnn_shim = True
    if not hasattr(np, "float"):
        np.float = float
    try:
        import pandas as pd
        if not getattr(pd.DataFrame, "_stemgnn_shim", False):
            _orig_fillna = pd.DataFrame.fillna

            def _fillna(self, value=None, *a, method=None, limit=None, **kw):
                if method == "ffill":
                    return self.ffill(limit=limit)
                if method == "bfill":
                    return self.bfill(limit=limit)
                return _orig_fillna(self, value, *a, **kw)

            pd.DataFrame.fillna = _fillna
            pd.DataFrame._stemgnn_shim = True
    except ImportError:  # pandas only matters for the dataloader
        pass


@contextlib.contextmanager
def reference_modules():
    """Context manager: inside it `models`, `data_loader`, `utils` resolve to the REFERENCE
    packages (not this repo's drop-in packages of the same names).  On exit the repo's own
    modules are restored in sys.modules."""
    if not reference_available():
        raise RuntimeError(f"reference not found at {REFERENCE_ROOT!r} (set STEMGNN_REFERENCE_ROOT)")
    _install_patches()
    names = ("models", "data_loader", "utils")
    saved = {k: v for k, v in sys.modules.items()
             if k in names or any(k.startswith(n + ".") for n in names)}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        yield
    finally:
        sys.path.remove(REFERENCE_ROOT)
        for k in [k for k in sys.modules
                  if k in names or any(k.startswith(n + ".") for n in names)]:
            del sys.modules[k]
        sys.modules.update(saved)


def load_reference_model_class():
    """Returns the reference `models.base_model.Model` class (kept alive after the context)."""
    with reference_modules():
        mod = importlib.import_module("models.base_model")
        return mod.Model


def build_reference_model(units, time_step, multi_layer, horizon, seed=0, stack_cnt=2):
    """Reference Model under torch.manual_seed(seed) (main.py:52 uses seed 0), on CPU."""
    import torch
    cls = load_reference_model_class()
    torch.manual_seed(seed)
    return cls(units, stack_cnt, time_step, multi_layer, horizon=horizon)
