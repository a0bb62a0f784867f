#!/usr/bin/env python
"""bench.py — forecast-windows/sec of the StemGNN hot path on B200 (BASELINE.json metric).

A "step" is ONE pass of the hot path (Model.forward in eval(), no_grad — SURVEY.md §8(d)) over one
batch of windows per GPU (weak scaling: every rank owns its own batch; the eval path has no collective).
Default workload = BASELINE.json configs[1], the shape the metric is quoted on: (B,N,W,H)=(32,358,12,3).

    python bench.py [--gpus N --steps K --warmup W] [--config cfg1..cfg5]     # this repo's CUDA path
    python bench.py ... --dump-outputs DIR       # also write the last timed step's forecast / attention as DIR/*.npy
    python bench.py --impl reference [...]                                    # the reference's own CPU path

Prints ONE JSON line.  Keys (see the task contract):
  value / ms_per_step   device-timed (CUDA events, L2 flushed between steps), inputs resident in HBM
  e2e                   same metric through the public API with HOST buffers, per step inside the timed region: pinned x ->
                        H2D -> the captured forward -> D2H of the forecast -> synchronize, via Model.inference_session
                        (stemgnn_b200/session.py); `plain_forward_loop` = the same with x.to(dev) -> Model.forward
  parity                "MAE vs ref" half of the metric: utils.math_utils.MAE and allclose(rtol 1e-3, atol 1e-4)
                        between this forward and the reference's CPU forward on the SAME inputs/weights
  roofline              the dominant kernel (GRU recurrence), timed live with CUDA events via the
                        library's stemgnn_profile_gru hook; flops = SURVEY.md §8(d) GRU terms
  cpu_baseline          the unmodified reference (the checkout named by STEMGNN_REFERENCE_ROOT, under oracle/ref_shim.py;
                        kind "reference") — or the torch port when it is not set (kind "port") — on the host cores

Inputs and weights come from fixed seeds, so runs with the same arguments see identical inputs and two builds can be
compared output for output through --dump-outputs.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MULTI = 5
METRIC = "forecast-windows/sec (B,N,W)=(32,358,12)"
# BASELINE.json configs; B is per GPU (cfg4: global 128 on 4 GPUs, cfg5: global 256 on 8 GPUs)
CONFIGS = {
    "cfg1": dict(B=32, N=140, W=12, H=3, gemm="auto",
                 workload="synthetic N=140 W=12 H=3 batch=32 fp32 eval forward (BASELINE.json configs[0] shape)"),
    "cfg2": dict(B=32, N=358, W=12, H=3, gemm="auto",
                 workload="synthetic N=358 W=12 H=3 batch=32 fp32 eval forward (BASELINE.json configs[1])"),
    "cfg3": dict(B=64, N=228, W=12, H=3, gemm="bf16",
                 workload="PeMS07 shape N=228 W=12 H=3 batch=64 bf16 tensor-core GFT eval forward (BASELINE.json configs[2])"),
    "cfg4": dict(B=32, N=325, W=12, H=12, gemm="auto",
                 workload="synthetic N=325 W=12 H=12 batch=32 per GPU (global 128 on 4 GPUs) eval forward (BASELINE.json configs[3])"),
    "cfg5": dict(B=32, N=2048, W=12, H=3, gemm="auto",
                 workload="synthetic N=2048 W=12 H=3 batch=32 per GPU (global 256 on 8 GPUs) eval forward (BASELINE.json configs[4])"),
}


def config_dict(name, world):
    """The `config` object of the JSON line — identical for both arms (ours / --impl reference)."""
    c = CONFIGS[name]
    return {"workload": c["workload"], "name": name, "B_per_gpu": c["B"], "N": c["N"], "W": c["W"], "H": c["H"],
            "multi_layer": MULTI, "mode": "eval forward (Model.forward, no_grad)",
            "parallelism": f"dp{world} replicas"}


def _peaks():
    extra = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r02_measured_peaks_tf32_fp32.json")) as f:
            extra = json.load(f)
    except Exception:
        pass
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops"]), float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst)", extra
    except Exception:
        return 1590.0, 6650.0, "fallback (B200_PROFILING.md)", extra


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.  NVML is polled from a background thread
    every ~2 ms (the timed region is only tens of milliseconds long, too short for `nvidia-smi -lms`); falls back
    to one nvidia-smi query when pynvml is unavailable."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, index):
        import threading
        self.index, self.samples, self.reason_bits, self.max_mhz = index, [], 0, None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML indices follow the physical order; honour CUDA_VISIBLE_DEVICES when it lists integers
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                try:
                    phys = int(vis.split(",")[index])
                except (ValueError, IndexError):
                    phys = index
            self._nv, self._h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
        except Exception:
            self._nv = None

    def _poll(self):
        nv, h = self._nv, self._h
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
            sm = sorted(self.samples)
            reasons = sorted(k for k, bit in self.REASONS.items() if self.reason_bits & bit)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "nvml polled every 2 ms inside the timed region"}
        try:
            out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits",
                                  "-i", str(self.index)], capture_output=True, text=True, timeout=10).stdout
            f = [v.strip() for v in out.strip().split(",")]
            return {"sm_mhz": float(f[0]), "sm_max_mhz": float(f[1]), "reasons": [], "samples": 1,
                    "source": "nvidia-smi, one query right after the timed region"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0}


def make_inputs(name, rank):
    """(x (B,W,N), y (B,H,N), data tag): the seeded synthetic generator of SURVEY.md §8(d), seed 1234 + rank."""
    from stemgnn_b200 import synthetic
    c = CONFIGS[name]
    x, y = synthetic.synthetic_batch(c["B"], c["N"], c["W"], c["H"], seed=1234 + rank)
    return x, y, "synthetic"


def cpu_reference(name, budget_s=20.0, max_steps=15):
    """Times the reference's CPU forward on this host for `name`: (CpuReference, x, ms/forward, steps, threads)."""
    import torch
    from oracle.cpu_reference import CpuReference
    from stemgnn_b200 import synthetic
    c = CONFIGS[name]
    p = synthetic.synthetic_params(c["N"], c["W"], c["H"], MULTI, seed=0)
    ref = CpuReference(c["N"], c["W"], c["H"], MULTI, p)
    x, _y, _tag = make_inputs(name, 0)
    threads = ref.pick_threads(x, cands=None if c["N"] <= 512 else [min(32, os.cpu_count() or 8), os.cpu_count() or 8])
    t0 = time.perf_counter()
    ref.forward(x)
    one = time.perf_counter() - t0
    steps = max(1, min(max_steps, int(budget_s / max(one, 1e-3))))
    ms = ref.time_forward(x, steps, 1 if one < 2.0 else 0) * 1e3
    return ref, x, ms, steps, threads


def run_reference(args, rank, world):
    if rank != 0:
        return
    c = CONFIGS[args.config]
    ref, _x, ms, steps, threads = cpu_reference(args.config, budget_s=30.0, max_steps=max(1, min(args.steps, 40)))
    v = c["B"] / (ms * 1e-3)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "windows/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": make_inputs(args.config, 0)[2],
            "config": config_dict(args.config, world),
            "impl_notes": f"reference CPU path = {ref.kind} ({ref.source}), torch {__import__('torch').__version__} CPU, "
                          f"{threads} threads (best of a sweep)",
            "cpu_baseline": {"value": v, "unit": "windows/s", "cores": threads, "kind": ref.kind,
                             "sample": f"{steps} eval forwards of one {c['B']}-window batch; os.cpu_count()={os.cpu_count()}"},
            "e2e": {"value": v, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    from models.base_model import Model
    from stemgnn_b200 import synthetic as tp      # seeded weights / inputs (plain data generators)
    from stemgnn_b200 import _lib, runtime as _rt

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()
    cfg = CONFIGS[args.config]
    B, N, W, H = cfg["B"], cfg["N"], cfg["W"], cfg["H"]
    gemm_mode = {"auto": _rt.GEMM_AUTO, "bf16": getattr(_rt, "GEMM_BF16", _rt.GEMM_AUTO)}[cfg["gemm"]]

    model = Model(N, 2, W, MULTI, horizon=H)
    model.load_state_dict(tp.synthetic_params(N, W, H, MULTI, seed=0))
    model = model.to(dev).eval()
    model.gemm_mode = gemm_mode
    x_host, y_host, data_tag = make_inputs(args.config, rank)
    x_host = x_host.pin_memory()
    x_dev = x_host.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    steps = args.steps

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        # kernels per forward, counted on an eager forward (graph replays launch the same kernels, but the library's counter
        # only sees the launches it issues itself, i.e. the capture)
        model.use_cuda_graph = False
        model(x_dev); model(x_dev)
        c0 = lib.stemgnn_launch_count()
        model(x_dev)
        launches_per_forward = int(lib.stemgnn_launch_count() - c0)
        model.use_cuda_graph = True
        model(x_dev)                                  # captures the graph (synchronises the host) and uploads it
        # ---- device-timed: inputs resident in HBM, L2 flushed between steps -------------------
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(steps)]
        sampler = ClockSampler(local_rank) if rank == 0 else None
        barrier()
        # Every timed event pair must bracket device work only.  The stream is held for ~0.2 s by a spin kernel while the host
        # enqueues the warm-up and timed steps (~0.2 ms of host time each; beyond the launch queue's depth the host is that
        # queue ahead), and the warm-up runs back to back into the timed steps.  Otherwise a stall of the host thread
        # (measured on a B200 at 1000 W: 8 and 70 ms, from NVML queries and the shared host CPUs), or the ~0.2 ms to submit the first
        # step to an idle device, lands inside a timed step.
        torch.cuda._sleep(400_000_000)                # cycles: 0.2 s at 2 GHz
        for _ in range(max(args.warmup, 3)):
            flush.zero_()
            model(x_dev)
        for i in range(steps):
            flush.zero_()
            ev[i][0].record()
            f_dev, a_dev = model(x_dev)
            ev[i][1].record()
        barrier()
        launches = launches_per_forward * steps      # + 3 torch copy kernels per step around the graph replay
        clocks = sampler.stop() if sampler else None
        dev_ms = sum(a.elapsed_time(b) for a, b in ev)
        forecast_ours = f_dev.float().cpu()

        # ---- same forward with every GEMM forced to exact fp32 FFMA2 (Model.gemm_mode = 1) ---------------
        model.gemm_mode = _rt.GEMM_FP32
        for _ in range(3):
            model(x_dev)
        ev32 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                for _ in range(min(steps, 20))]
        for a0, a1 in ev32:
            flush.zero_()
            a0.record()
            model(x_dev)
            a1.record()
        torch.cuda.synchronize()
        fp32_ms = sum(a0.elapsed_time(a1) for a0, a1 in ev32) / len(ev32)
        model.gemm_mode = gemm_mode
        model(x_dev)

        # ---- dominant kernel (GRU recurrence) with CUDA events on the launching stream --------------
        gru_ms = None
        try:
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); e1.record(); torch.cuda.synchronize()           # materialise the handles
            tot = 0.0
            reps = min(steps, 10)
            model.use_cuda_graph = False          # the event hook lives inside the C call: eager launches for this measurement
            model(x_dev)
            for _ in range(reps):
                flush.zero_()
                lib.stemgnn_profile_gru(e0.cuda_event, e1.cuda_event)
                model(x_dev)
                lib.stemgnn_profile_gru(None, None)
                torch.cuda.synchronize()
                tot += e0.elapsed_time(e1)
            gru_ms = tot / reps
            model.use_cuda_graph = True
        except Exception as exc:                                        # hook is optional evidence
            gru_ms = None
            sys.stderr.write(f"[bench] GRU event hook failed: {exc}\n")

        # ---- the fused tcgen05 GLU chain (61 % of the flops), timed alone through the C ABI ------------------
        glu_ms, glu_flops = None, None
        try:
            glu_ms, glu_flops = time_glu_chain(lib, dev, B, N, W, flush)
        except Exception as exc:
            sys.stderr.write(f"[bench] GLU chain timing failed: {exc}\n")

        # ---- end to end through the public API with host buffers ----------------------------------
        # public API for host buffers: Model.inference_session(B) — per call: H2D of the batch into the captured graph's static
        # input, ONE graph replay of the forward, D2H of the forecast (stemgnn_b200/session.py).  Also timed: the plain
        # `model(x_host.to(dev))` loop (the reference's inference loop shape, handler.py:34-40), reported beside it.
        out_host = torch.empty(B, H, N).pin_memory()
        for _ in range(3):
            f, _a = model(x_host.to(dev, non_blocking=True))
            out_host.copy_(f, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            xd = x_host.to(dev, non_blocking=True)                      # H2D of the step's input
            f, _a = model(xd)
            out_host.copy_(f, non_blocking=True)                        # D2H of the step's result
            torch.cuda.synchronize()
        e2e_plain_s = time.perf_counter() - t0
        sess = model.inference_session(B)
        for _ in range(3):
            sess(x_host, out_host)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            sess(x_host, out_host)                                      # H2D + graph replay + D2H, stream-ordered
            torch.cuda.synchronize()                                    # the step's result is on the host
        e2e_s = time.perf_counter() - t0
        barrier()
        e2e_forecast = out_host.clone()
        sys.stderr.write(f"[bench] e2e session {e2e_s / steps * 1e3:.3f} ms/step, plain Model.forward loop "
                         f"{e2e_plain_s / steps * 1e3:.3f} ms/step\n")

    # ---- second column: training step (handler.py:160-165) ----------------------------------------------
    train = None
    try:
        train = time_train_step(model, x_dev, y_host.to(dev), flush, barrier, steps, world)
    except Exception as exc:
        sys.stderr.write(f"[bench] train-step timing failed: {exc}\n")
    model.eval()

    train_ms = train["total_ms"] if train else 0.0
    t = torch.tensor([dev_ms, e2e_s * 1e3, train_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, train_ms = float(t[0]), float(t[1]), float(t[2])
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, forecast=f_dev, attention=a_dev)

    peak_tf, peak_gbs, peak_src, extra_peaks = _peaks()
    gru_flops = 6.0 * B * N ** 3 + 12.0 * B * N * N               # SURVEY §8(d): recurrence + gates
    roof = None
    if gru_ms and N > 512:
        # cfg5 envelope: W_hh does not fit on chip; every step streams its fp16 hi/lo images (2 x 3N x N x 2 bytes) plus the
        # h tile of every CTA from L2/HBM -> the recurrence is bandwidth-bound (DESIGN.md §5, gru_step_tc.cu)
        nt, kp = (N + 39) // 40, (N + 63) // 64 * 64
        step_bytes = 2.0 * nt * 128 * kp * 2 + nt * ((B + 31) // 32) * 64 * kp * 2
        ach = step_bytes * N / (gru_ms * 1e-3) / 1e9
        roof = {"kernel": "gru_step_tc_kernel x N launches (tcgen05 kind::f16, W_hh hi/lo images streamed by TMA)",
                "bound": "hbm", "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs, "traffic": None,
                "peak_source": peak_src + " (copy bandwidth; the 50 MB image set is L2-resident, so this is a lower bound "
                                          "on the applicable peak)",
                "ms_per_launch": gru_ms / N, "launches": N, "share_of_step": gru_ms / (dev_ms / steps),
                "algorithmic_bytes_per_launch": step_bytes, "algorithmic_flops_per_forward": gru_flops,
                "measured_other_peaks": extra_peaks,
                "note": f"{N} dependent steps, one launch each; bytes = W_hh hi/lo images + per-CTA h tiles per step"}
    elif gru_ms:
        ach = gru_flops / (gru_ms * 1e-3) / 1e12
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "r02_gru_traffic.json")) as f:
                tj = json.load(f)
            if tj.get("config") == args.config:
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            pass
        roof = {"kernel": lib.stemgnn_gru_kernel_name().decode() if hasattr(lib, "stemgnn_gru_kernel_name") else "gru",
                "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram__bytes_read+write of profiles/r02_gru_traffic.json)"
                if traffic else None,
                "peak_source": peak_src, "ms_per_launch": gru_ms, "share_of_step": gru_ms / (dev_ms / steps),
                "algorithmic_flops_per_launch": gru_flops, "measured_other_peaks": extra_peaks,
                "note": f"recurrence of {N} dependent steps (latency chain: exchange -> 2*ceil(N/16) MMAs -> gates per step); "
                        "flops = 6BN^3 + 12BN^2 counted once (SURVEY.md §8(d)), the split-operand kernel issues 4x of them"}

    # ---- parity: "MAE vs ref" on the SAME inputs / weights, reference CPU forward timed beside it ----------------
    ref, x_ref, cpu_ms, cpu_steps, threads = cpu_reference(args.config)
    f_ref, _a_ref = ref.forward(x_ref)
    err = (forecast_ours.double() - f_ref.double()).abs()
    parity = {"mae_vs_ref": float(err.mean()), "max_abs_err": float(err.max()),
              "allclose_rtol1e-3_atol1e-4": bool((err <= 1e-4 + 1e-3 * f_ref.double().abs()).all()),
              "ref": ref.kind, "ref_source": ref.source,
              "what": "utils.math_utils.MAE / allclose between this run's timed forecast (rank 0) and the reference CPU forward"}
    cpu_v = B / (cpu_ms * 1e-3)
    value = world * B * steps / (dev_ms * 1e-3)
    prec = {"auto": "f32 (GLU chain / GFT / output map on tcgen05 with split operands, fp32 accumulate; see exact_fp32)",
            "bf16": "bf16 tensor-core operands (GLU chain, GFT), fp32 accumulate"}[cfg["gemm"]]
    line = {"metric": METRIC, "value": value, "unit": "windows/s", "n_gpus": world, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": prec, "data": data_tag,
            "exact_fp32": {"value": B / (fp32_ms * 1e-3) * world, "unit": "windows/s", "ms_per_step": fp32_ms,
                           "what": "same forward with every GEMM on the fp32 FFMA2 path (Model.gemm_mode = 1), rank 0"},
            "config": config_dict(args.config, world),
            "impl_notes": {"l2": "flushed between timed steps (256 MiB memset outside the event pairs)",
                           "reuse_folded": "eval forwards reuse the DFT-folded / pre-split weights while no parameter "
                                           "changed (weight pre-packing, stemgnn_fwd_opts_t.reuse_folded)",
                           "cuda_graph": "with frozen weights Model.forward replays one captured CUDA graph of its launches "
                                         "(input copied into / outputs cloned out of static buffers, inside the timed region)",
                           "flops_per_step": forward_flops(B, N, W, H)},
            "parity": parity,
            "e2e": {"value": world * B * steps / (e2e_ms * 1e-3), "unit": "windows/s",
                    "h2d_bytes_per_step": B * W * N * 4, "d2h_bytes_per_step": B * H * N * 4,
                    "ms_per_step": e2e_ms / steps,
                    "api": "Model.inference_session(B)(x_pinned, out_pinned) + torch.cuda.synchronize() per step: H2D of the batch, "
                           "one CUDA-graph replay, D2H of the forecast",
                    "max_abs_diff_vs_device_timed_forecast": float((e2e_forecast - forecast_ours).abs().max()),
                    "plain_forward_loop": {"value": B * steps / e2e_plain_s, "unit": "windows/s (rank 0)",
                                           "ms_per_step": e2e_plain_s / steps * 1e3,
                                           "what": "x_host.to(dev) -> model(x) -> out_host.copy_(forecast) -> synchronize "
                                                   "(Model.forward re-validates ~70 parameter pointers / versions per call)"}},
            "train": None if not train else {
                "value": world * B * train["steps"] / (train_ms * 1e-3), "unit": "windows/s",
                "ms_per_step": train_ms / train["steps"], "steps": train["steps"], "what": train["what"]},
            "gpu_launches": int(launches),
            "roofline": roof,
            "roofline_glu": None if not glu_ms else {
                "kernel": "glu_chain_h_kernel<SPLIT> (tcgen05 kind::f16, fp16 hi/lo split operands: 3 MMAs per product; the 3 GLU "
                          "layers of one chain over B*N rows) + its operand-split pre-pass (7 small launches: G and 6 weights)",
                "bound": "tensor", "achieved": glu_flops / (glu_ms * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": glu_flops / (glu_ms * 1e-3) / 1e12 / peak_tf, "ms_per_launch": glu_ms,
                "algorithmic_flops_per_launch": glu_flops, "peak_source": peak_src,
                "note": "L2 flushed before each launch: weights and the G tile come from HBM"},
            "cpu_baseline": {"value": cpu_v, "unit": "windows/s", "cores": threads, "kind": ref.kind,
                             "sample": f"{cpu_steps} eval forwards of one {B}-window batch "
                                       f"({cpu_ms:.1f} ms each); os.cpu_count()={os.cpu_count()}"},
            "clocks": clocks}
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, **arrays):
    """What a caller of the timed forward receives — Model.forward's (forecast (B,H,N), attention (N,N)) — as
    float32 <out_dir>/<name>.npy.  The largest configuration writes 17 MB (cfg5: attention 2048 x 2048)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def forward_flops(B, N, W, H, S=2, K=4):
    """SURVEY.md §8(d) dead-work-free forward flops."""
    T = MULTI * W
    d = K * T
    blk = (2 * (K - 1) * B * N * N * W + 2 * B * N * d * 2 * (36 + 30) * W / 12 + 2 * B * N * d * d * 4 +
           2 * B * N * d * 2 * (124 + 116) * T / 60 + 2 * K * B * N * T * T + 2 * B * N * (T * T + T * W))
    return float(6 * B * N * N * W + 6 * B * N ** 3 + 12 * B * N * N + 10 * B * N * N + 4 * N ** 3 + 6 * N * N +
                 S * blk + 2 * B * N * (T * W + W * W) + 2 * B * N * (W * W + W * H))


def time_glu_chain(lib, dev, B, N, W, flush):
    """One launch of the fused 3-layer GLU chain kernel (K1 = 3W -> d -> d -> d over B*N rows), CUDA events."""
    import torch
    if not hasattr(lib, "stemgnn_glu_chain"):
        return None, None
    R, d, K1 = B * N, 4 * MULTI * W, 3 * W
    g = torch.Generator().manual_seed(5)
    G = torch.randn(R, K1, generator=g).to(dev)
    ws = [torch.randn(d, K1 if l == 0 else d, generator=g).div_((K1 if l == 0 else d) ** 0.5).to(dev)
          for l in range(3) for _ in range(2)]
    bs = [torch.zeros(d, device=dev) for _ in range(6)]
    out = torch.empty(R, d, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    wp = (ctypes.c_void_p * 6)(*[t.data_ptr() for t in ws])
    bp = (ctypes.c_void_p * 6)(*[t.data_ptr() for t in bs])
    scratch = torch.empty(int(lib.stemgnn_glu_chain_scratch_bytes(R, d, K1)), dtype=torch.uint8, device=dev)

    def call():
        rc = lib.stemgnn_glu_chain(R, d, K1, G.data_ptr(), K1, wp, bp, out.data_ptr(), d, 0, scratch.data_ptr(), st)
        if rc:
            raise RuntimeError(lib.stemgnn_last_error().decode())
    for _ in range(3):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tot, reps = 0.0, 10
    for _ in range(reps):
        flush.zero_()
        e0.record(); call(); e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    flops = 2.0 * R * 2 * d * (K1 + d + d)          # algorithmic: one product per element pair (the split issues 3)
    return tot / reps, flops


def time_train_step(model, x_dev, y_dev, flush, barrier, steps, world):
    """zero_grad + forward (train mode, Philox dropout) + MSE + backward (+ the single flat-gradient all-reduce
    at N>1) + RMSprop: through the captured-graph trainer when the package has one, else eager torch."""
    import torch
    from stemgnn_b200 import ddp
    ddp.attach(model)
    model.train()
    what = "zero_grad + forward(train, Philox dropout) + MSE + backward" + \
        (" + flat-gradient NCCL all-reduce" if world > 1 else "") + " + RMSprop step"
    try:
        from stemgnn_b200.trainer import FusedTrainer
        tr = FusedTrainer(model, optimizer="RMSProp", lr=1e-4)
        step = lambda: tr.step(x_dev, y_dev)                       # noqa: E731
        what += " — one CUDA graph replay (stemgnn_b200.trainer.FusedTrainer, fused RMSprop kernel, no host sync)"
    except ImportError:
        optim = torch.optim.RMSprop(model.parameters(), lr=1e-4, eps=1e-8)
        crit = torch.nn.MSELoss()

        def step():
            model.zero_grad()
            f, _a = model(x_dev)
            loss = crit(f, y_dev)
            loss.backward()
            optim.step()
    t_steps = max(5, min(steps, 20))
    for _ in range(3):
        step()
    tev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(t_steps)]
    barrier()
    for i in range(t_steps):
        flush.zero_()
        tev[i][0].record()
        step()
        tev[i][1].record()
    barrier()
    return {"total_ms": sum(a.elapsed_time(b) for a, b in tev), "steps": t_steps, "what": what}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's forecast and attention (rank 0) to DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
