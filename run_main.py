#!/usr/bin/env python
"""Runs the UNMODIFIED reference `main.py` against this repo's drop-in `models/`, `data_loader/`,
`utils/` packages (SURVEY.md §8(b) "Launching the unchanged main.py").

    STEMGNN_REFERENCE_ROOT=<checkout> python run_main.py --device cuda:0 --epoch 1 [--dataset ECG_data ...]   # any main.py flag

`main.py` does `from models.handler import train, test`; run as a script it would import the
reference's own packages, so this launcher puts the repo first on sys.path and executes the
reference file with runpy.  It runs from a scratch cwd holding a `dataset` symlink (main.py uses
cwd-relative `dataset/<name>.csv` and writes `output/`).  Note main.py:3 pins
CUDA_VISIBLE_DEVICES='0,1'; multi-GPU training beyond that goes through `stemgnn_b200.ddp`.
"""
import os
import runpy
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))


REF = os.environ.get("STEMGNN_REFERENCE_ROOT", "")       # a microsoft/StemGNN checkout


def main():
    ref_main = os.path.join(REF, "main.py")
    if not REF or not os.path.exists(ref_main):
        raise SystemExit(f"reference main.py not found at {ref_main} (set STEMGNN_REFERENCE_ROOT)")
    work = os.environ.get("STEMGNN_WORKDIR", os.path.join(ROOT, "gpurun_out", "main_run"))
    os.makedirs(work, exist_ok=True)
    link = os.path.join(work, "dataset")
    if not os.path.exists(link):
        os.symlink(os.path.join(REF, "dataset"), link)
    os.chdir(work)
    sys.path.insert(0, ROOT)
    sys.argv = [ref_main] + sys.argv[1:]
    runpy.run_path(ref_main, run_name="__main__")


if __name__ == "__main__":
    main()
