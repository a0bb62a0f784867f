"""TEST / BENCH INFRASTRUCTURE — not product code.

The reference's own CPU implementation of the hot path, ready to call: the UNMODIFIED reference
`models.base_model.Model` (the checkout named by STEMGNN_REFERENCE_ROOT) imported under the 4-patch shim
of oracle/ref_shim.py, with the same seeded weights the CUDA model is loaded with.  When it is not set the
torch port (oracle/torch_port.py, the same ATen op sequence) stands in and says so.

Only `bench.py` (`--impl reference`, `cpu_baseline`, the MAE-vs-ref parity figure) and `oracle/make_golden.py`
import this.
"""
import os
import time

import torch

from . import ref_shim, torch_port as tp


class CpuReference:
    """forward(x (B,W,N) cpu) -> (forecast (B,H,N), attention (N,N)), eval mode, no_grad."""

    def __init__(self, N, W, H, multi, params):
        self.kind = "port"
        self.params = {k: v.detach().cpu().float() for k, v in params.items()}
        self.model = None
        if ref_shim.reference_available():
            cls = ref_shim.load_reference_model_class()
            m = cls(N, 2, W, multi, horizon=H)
            m.load_state_dict(self.params, strict=True)
            self.model = m.eval()
            self.kind = "reference"
        self.source = ref_shim.REFERENCE_ROOT if self.model is not None else "oracle/torch_port.py"

    def forward(self, x):
        with torch.no_grad():
            if self.model is not None:
                return self.model(x)
            return tp.model_forward(x, self.params)

    def pick_threads(self, x, cands=None):
        """torchrun pins OMP_NUM_THREADS=1 and "all cores" is not the fastest setting on a 128-thread host:
        the reference gets its best shot from a short sweep.  Returns the chosen thread count."""
        ncpu = os.cpu_count() or 8
        cands = cands or sorted({c for c in (8, 16, 32, 64, ncpu // 2, ncpu) if 1 <= c <= ncpu})
        best, best_t = cands[0], None
        for c in cands:
            torch.set_num_threads(c)
            self.forward(x)
            t0 = time.perf_counter()
            self.forward(x)
            dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best, best_t = c, dt
        torch.set_num_threads(best)
        return best

    def time_forward(self, x, steps, warmup):
        for _ in range(warmup):
            self.forward(x)
        t0 = time.perf_counter()
        for _ in range(steps):
            self.forward(x)
        return (time.perf_counter() - t0) / steps
