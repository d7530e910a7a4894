"""Device resampling (septfa_resample) at the batched-file workload: 256 mixtures of 4 s at 44.1 and 48 kHz, float32 and
int16 input, to 16 kHz.

Each case is timed with CUDA events over --iters back-to-back calls after --warmup calls. The inputs (98 .. 197 MB)
and outputs (65.5 MB) exceed the 126 MB L2 together, so every call streams from HBM. The kernel's least traffic is one
read of the input and one write of the output; the record gives that over the measured time, as a fraction of the HBM
data-sheet rate (7.7 TB/s) and of the rate this project measured for a plain copy kernel (6.55 TB/s). The kernel does
2 x (taps per output) flops per output: at ~40 .. 110 taps that is 5 .. 14 GFLOP per call, far under the fp32 rate, so
HBM is the bound that applies; the record says so when the time is within 2x of the HBM floor, and "not at the HBM
bound" otherwise.

With --to it times the output direction instead (septfa_resample_to): the separated output of a 256 x 4 s forward,
[512, 64000] float32 at 16 kHz, to 44.1 and 48 kHz (131 MB in, 360 / 393 MB out), with the same fields.

    python tools/resample_bench.py [--iters 50 --warmup 5] [--to] --out FILE.json
"""
import argparse
import contextlib
import ctypes as C
import io
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from septfa_b200 import lib as _lib  # noqa: E402
from septfa_b200 import synth  # noqa: E402
from septfa_b200.model import SeparationModel  # noqa: E402

HBM_DATASHEET = 7.7e12
HBM_MEASURED = 6.55e12


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = ([v.strip() for v in q.stdout.strip().split(",")] + [None] * 3)[:3]
    return {"gpu": name or torch.cuda.get_device_name(index), "power_limit": power, "sm_max_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--seconds", type=float, default=4.0)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--to", action="store_true", help="time septfa_resample_to on the output of a --batch x --seconds forward")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("resample_bench measures on a CUDA device; none found")
    dev = torch.device("cuda", 0)
    with contextlib.redirect_stdout(io.StringIO()):
        model = SeparationModel(**synth.CONFIG_WITH_VAD)
    model.eval().to(dev)
    h = model._handle(dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    cases = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(call):
        for _ in range(a.warmup):
            call()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(a.iters):
            call()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / a.iters / 1e3

    for rate in (44100, 48000) if a.to else ():
        rows, L16 = 2 * a.batch, int(round(a.seconds * 16000))   # both speakers of every mixture
        L = -(-rate * L16 // 16000)
        y = torch.rand((rows, L16), generator=torch.Generator(device=dev).manual_seed(rate), device=dev) * 1.8 - 0.9
        out = torch.empty((rows, L), device=dev)
        t = timed(lambda: _lib.check(h.ptr, h.lib.septfa_resample_to(h.ptr, C.c_void_p(y.data_ptr()), rows, L16, rate,
                                                                     C.c_void_p(out.data_ptr()), stream)))
        nbytes = y.numel() * 4 + out.numel() * 4
        floor = nbytes / HBM_DATASHEET
        gcd = math.gcd(rate, 16000)
        cases.append({"rate": rate, "direction": "16000 -> rate", "rows": rows, "L16": L16, "L": L,
                      "orig": 16000 // gcd, "new": rate // gcd, "delay": _lib.resample_to_geometry(rate)[0],
                      "kernel_us": t * 1e6, "bytes": nbytes, "achieved_TBps": nbytes / t / 1e12,
                      "of_hbm_datasheet": floor / t, "of_hbm_measured": (nbytes / HBM_MEASURED) / t,
                      "hbm_floor_measured_us": nbytes / HBM_MEASURED * 1e6,
                      "bound": "HBM" if t < 2 * floor else "not at the HBM bound"})
    for rate in () if a.to else (44100, 48000):
        L = int(round(a.seconds * rate))
        L16 = -(-16000 * L // rate)
        g = torch.Generator(device=dev).manual_seed(rate)
        xf = torch.rand((a.batch, L), generator=g, device=dev) * 1.8 - 0.9
        for fmt, x in (("f32", xf), ("pcm16", (xf * 32000).to(torch.int16))):
            out = torch.empty((a.batch, L16), device=dev)
            x_fmt = _lib.FMT_PCM16 if fmt == "pcm16" else _lib.FMT_F32

            def call():
                _lib.check(h.ptr, h.lib.septfa_resample(h.ptr, C.c_void_p(x.data_ptr()), x_fmt, a.batch, L, rate,
                                                         C.c_void_p(out.data_ptr()), stream))
            t = timed(call)
            nbytes = x.numel() * x.element_size() + out.numel() * 4
            floor = nbytes / HBM_DATASHEET
            gcd = math.gcd(rate, 16000)
            cases.append({"rate": rate, "input": fmt, "batch": a.batch, "L": L, "L16": L16,
                          "orig": rate // gcd, "new": 16000 // gcd, "delay": _lib.resample_geometry(rate)[0],
                          "kernel_us": t * 1e6, "bytes": nbytes, "achieved_TBps": nbytes / t / 1e12,
                          "of_hbm_datasheet": floor / t, "of_hbm_measured": (nbytes / HBM_MEASURED) / t,
                          "bound": "HBM" if t < 2 * floor else "not at the HBM bound"})
    rec = {"bench": "septfa_resample_to" if a.to else "septfa_resample", **gpu_info(0),
           "timing": f"CUDA events over {a.iters} back-to-back calls after {a.warmup} warm-up calls",
           "hbm_datasheet_TBps": HBM_DATASHEET / 1e12, "hbm_measured_copy_TBps": HBM_MEASURED / 1e12, "cases": cases}
    print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
