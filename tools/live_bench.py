"""Live-session push latency against the lockstep online step at the same number of streams.

Workload: a live session of --capacity slots (config_with_vad, seeded weights, filter_signals_by_smo_vad). Slot s starts
its first stream at step s mod 7; every stream runs 3 .. 10 hops of a seeded synthetic mixture, then its slot releases
and starts the next stream at the same step. Once all slots have started, every step pushes every slot (n = capacity),
with some slots at k = 0 .. 2 (zero-padded windows) and the rest in steady state. The lockstep leg is
septfa_online_step on the same number of streams with resident 3 s windows (the online leg of bench.py). The two legs
alternate step by step; each call is timed with CUDA events between two device synchronisations, on its own.

    python tools/live_bench.py [--capacity 1024 --steps 60 --warmup 10] --out profiles/live_bench_n1024.json
"""
import argparse
import contextlib
import ctypes as C
import io
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from septfa_b200 import lib as _lib  # noqa: E402
from septfa_b200 import synth  # noqa: E402
from septfa_b200.model import SeparationModel  # noqa: E402

HOP = 16000


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = ([v.strip() for v in q.stdout.strip().split(",")] + [None] * 3)[:3]
    return {"gpu": name or torch.cuda.get_device_name(index), "power_limit": power, "sm_max_clock": clock}


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(q * len(v)))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--capacity", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=60, help="timed steps per leg")
    ap.add_argument("--warmup", type=int, default=10, help="untimed steps first (>= 7: every slot has started)")
    ap.add_argument("--out", default=None, help="write the JSON record here too")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("live_bench measures on a CUDA device; none found")
    dev = torch.device("cuda", 0)
    args = synth.CONFIG_WITH_VAD
    with contextlib.redirect_stdout(io.StringIO()):
        model = SeparationModel(**args)
    model.load_state_dict(synth.make_state_dict(args, 41), strict=True)
    model.eval().to(dev)
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    ikw = _lib.InferKw.from_dict(kw)
    h = model._handle(dev)
    lib = h.lib
    n = a.capacity
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    # 32 distinct mixtures of 10 hops; stream j of slot s plays mixture (s + 7 j) % 32 for 3 + (s + j) % 8 hops
    mixes = torch.from_numpy(synth.make_mixtures(32, 10 * HOP, 4321)).to(dev).view(32, 10, HOP)
    start = np.arange(n) % 7
    gen = np.zeros(n, dtype=np.int64)          # streams finished per slot
    k = np.zeros(n, dtype=np.int64)            # hops pushed by the slot's current stream

    lv = C.c_void_p()
    _lib.check(h.ptr, lib.septfa_live_create(h.ptr, n, C.byref(lv)))
    ws = torch.empty(lib.septfa_live_workspace_bytes(lv, n), dtype=torch.uint8, device=dev)
    out = torch.empty((n, 2, HOP), device=dev)
    vad = torch.empty((n, 2, 63), device=dev)
    perm = torch.empty((n, 2), dtype=torch.int32, device=dev)

    st = C.c_void_p()
    _lib.check(h.ptr, lib.septfa_online_create(h.ptr, n, C.byref(st)))
    ws_on = torch.empty(lib.septfa_online_workspace_bytes(st), dtype=torch.uint8, device=dev)
    win = torch.from_numpy(np.tile(synth.make_mixtures(16, 48000, 4321), ((n + 15) // 16, 1))[:n]).to(dev)
    emitted = torch.empty((n, 2, HOP), device=dev)
    perm_on = torch.empty((n, 2), dtype=torch.int32, device=dev)

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    push_ms, step_ms, ns, restarts, launches = [], [], [], [], 0
    for t in range(a.warmup + a.steps):
        length = 3 + (np.arange(n) + gen) % 8
        ended = np.nonzero((k == length) & (start <= t))[0].astype(np.int32)
        if ended.size:
            _lib.check(h.ptr, lib.septfa_live_release(lv, ended.ctypes.data_as(C.c_void_p), ended.size, stream))
            gen[ended] += 1
            k[ended] = 0
        slots = np.nonzero(start <= t)[0].astype(np.int32)
        rng = np.random.default_rng(t)
        rng.shuffle(slots)
        mix = torch.from_numpy((slots + 7 * gen[slots]) % 32).to(dev)
        hops = mixes[mix, torch.from_numpy(k[slots]).to(dev)].contiguous()
        sl = slots.ctypes.data_as(C.c_void_p)

        def push():
            _lib.check(h.ptr, lib.septfa_live_push(lv, sl, slots.size, C.c_void_p(hops.data_ptr()), C.byref(ikw),
                                                   C.c_void_p(out.data_ptr()), C.c_void_p(vad.data_ptr()),
                                                   C.c_void_p(perm.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(), stream))

        def step():
            _lib.check(h.ptr, lib.septfa_online_step(st, C.c_void_p(win.data_ptr()), C.byref(ikw), C.c_void_p(emitted.data_ptr()),
                                                     C.c_void_p(perm_on.data_ptr()), C.c_void_p(ws_on.data_ptr()), ws_on.numel(),
                                                     stream))
        tp = timed(push)
        launches = lib.septfa_last_launch_count(h.ptr)
        ts = timed(step)
        k[slots] += 1
        if t >= a.warmup:
            assert slots.size == n, "timed steps must push every slot"
            push_ms.append(tp)
            step_ms.append(ts)
            ns.append(int(slots.size))
            restarts.append(int(ended.size))
    lib.septfa_live_destroy(lv)
    lib.septfa_online_destroy(st)

    p50p, p50s = pct(push_ms, 0.5), pct(step_ms, 0.5)
    rec = {"bench": "live_push_vs_lockstep_online_step", **gpu_info(0),
           "config": "config_with_vad, seeded weights, filter_signals_by_smo_vad, 3 s windows / 1 s hops",
           "streams": n, "timed_steps": len(push_ms), "warmup_steps": a.warmup,
           "releases_per_step_mean": float(np.mean(restarts)),
           "push": {"p50_ms": p50p, "p99_ms": pct(push_ms, 0.99), "min_ms": min(push_ms), "launches": launches},
           "lockstep_step": {"p50_ms": p50s, "p99_ms": pct(step_ms, 0.99), "min_ms": min(step_ms)},
           "push_over_step_p50": p50p / p50s,
           "timing": "CUDA events around one call between device synchronisations; legs alternate step by step",
           "state_bytes_per_slot": 4 + 6 * HOP * 4}
    line = json.dumps(rec)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
