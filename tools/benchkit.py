"""What the measurement tools in this directory share: the repository paths, the card readout, resident scenes,
CUDA-event windows, and the --reps / --out command line with the ending it implies.

The tools run as `python tools/<name>.py`, so `import benchkit` finds this module.  Importing it puts the repository
root and tests/ on sys.path (the tools reuse the tests' oracle bindings and helpers).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

from helpers import upload  # noqa: E402
from raytracing_c_b200 import driver, gpu_lib  # noqa: E402
from raytracing_c_b200._ffi import gpu_check  # noqa: E402


def card() -> dict:
    """The card's name, power limit and maximum SM clock: read in the run whose numbers they go with."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in out[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def init():
    """The GPU library with device 0 initialised; call it once per run."""
    gpu = gpu_lib()
    gpu_check(gpu.rt_gpu_init(0))
    return gpu


def resident(model: str, **kwargs) -> driver.LoadedScene:
    """assets/models/<model> loaded with the GPU library's callbacks (`kwargs` go to driver.load_scene), the callbacks
    registered and the scene uploaded."""
    loaded = driver.load_scene(os.path.join(ROOT, "assets", "models", model), **kwargs)
    upload(loaded)
    return loaded


def window_ms(fn, stream) -> float:
    """Milliseconds between two CUDA events recorded on `stream` around fn(), read after a device synchronise."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def per_call_ms(fn, stream, reps: int) -> float:
    """window_ms over `reps` back-to-back calls of fn, divided by `reps`.  Callers warm up and synchronise first, so the
    window opens on an idle stream."""
    def calls():
        for _ in range(reps):
            fn()
    return window_ms(calls, stream) / reps


def parser(reps: int) -> argparse.ArgumentParser:
    """The --reps / --out command line; a tool adds its own options to it."""
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=reps)
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    return ap


def finish(args, result: dict, summary, *scenes) -> None:
    """The ending of a run: one line with the card and the `summary` keys of `result`, `result` written to --out, the
    scenes closed, and exit status 1 when `result` holds a failed parity check."""
    print(json.dumps({"card": result["card"], **{k: result[k] for k in summary}}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    for s in scenes:
        s.close()
    if not result.get("parity_ok", True):
        sys.exit(1)
