"""Live-session push latency against the lockstep online step at the same number of streams and the same geometry.

Workload: a live session of --capacity slots with a window of --window and a hop of --hop samples (config_with_vad,
seeded weights, filter_signals_by_smo_vad). With c = window / (3 hop) (1 at the default 48000 / 16000), slot s starts
its first stream at step s mod 7c; every stream runs 3c .. 10c hops of a seeded synthetic mixture, then its slot
releases and starts the next stream at the same step. Once all slots have started, every step pushes every slot
(n = capacity), with some slots in their zero-padded first pushes and the rest in steady state. The lockstep leg is
septfa_online_step on the same number of streams with resident windows of the same geometry (the online leg of
bench.py at the default). The two legs alternate step by step; each call is timed with CUDA events between two device
synchronisations, on its own. realtime_streams = capacity * (hop / 16000) / push p99: the streams one GPU keeps up
with when it does nothing but push.

With --rate R (other than 16000) a third leg pushes the same schedule into a session at R Hz (septfa_live_create_rate):
every hop carries hop * R / 16000 native samples of seeded mixtures, which the session resamples on the device before
the same window / forward / emit. The three legs alternate step by step; the record adds the rate leg's push times and
its overhead over the 16 kHz push.

With --out-rate R (other than 16000) one more leg pushes the same schedule into a session at --rate in and R out
(septfa_live_create_rates), alternated step by step with the same session at 16 kHz out (the rate leg, or the 16 kHz
push when --rate is 16000); the record adds its push times and its overhead over that session.

    python tools/live_bench.py [--capacity 1024 --steps 60 --warmup 10c --window 48000 --hop 16000 --rate 48000
                                --out-rate 48000] --out FILE.json
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

FS = 16000


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
    ap.add_argument("--warmup", type=int, default=None, help="untimed steps first (default 10c; >= 7c: every slot has started)")
    ap.add_argument("--window", type=int, default=48000, help="window W in samples")
    ap.add_argument("--hop", type=int, default=16000, help="hop H in samples")
    ap.add_argument("--rate", type=int, default=16000, help="input rate of a third leg (16000: no third leg)")
    ap.add_argument("--out-rate", type=int, default=16000, help="output rate of one more leg (16000: no such leg)")
    ap.add_argument("--out", default=None, help="write the JSON record here too")
    a = ap.parse_args()
    W, H = a.window, a.hop
    c = W / (3 * H)                                  # hop counts scale with W / H
    period, max_hops = max(1, round(7 * c)), round(10 * c)
    if a.warmup is None:
        a.warmup = round(10 * c)
    if a.warmup < period:
        raise SystemExit(f"--warmup must be >= {period}: every slot must have started before the timed steps")
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

    # 32 distinct mixtures of 10c hops; stream j of slot s plays mixture (s + 7 j) % 32 for (3 + (s + j) % 8) c hops
    mixes = torch.from_numpy(synth.make_mixtures(32, max_hops * H, 4321)).to(dev).view(32, max_hops, H)
    start = np.arange(n) % period
    gen = np.zeros(n, dtype=np.int64)          # streams finished per slot
    k = np.zeros(n, dtype=np.int64)            # hops pushed by the slot's current stream

    lv = C.c_void_p()
    _lib.check(h.ptr, lib.septfa_live_create_win(h.ptr, n, W, H, C.byref(lv)))
    n_vad = lib.septfa_live_vad_frames(lv, None)
    ws = torch.empty(lib.septfa_live_workspace_bytes(lv, n), dtype=torch.uint8, device=dev)
    out = torch.empty((n, 2, H), device=dev)
    vad = torch.empty((n, 2, n_vad), device=dev)
    perm = torch.empty((n, 2), dtype=torch.int32, device=dev)

    lv_r = C.c_void_p()
    if a.rate != FS:
        _lib.check(h.ptr, lib.septfa_live_create_rate(h.ptr, n, W, H, a.rate, C.byref(lv_r)))
        delay = C.c_int()
        Hn = lib.septfa_live_input_hop(lv_r, C.byref(delay))
        ws_r = torch.empty(lib.septfa_live_workspace_bytes(lv_r, n), dtype=torch.uint8, device=dev)
        mixes_r = torch.from_numpy(synth.make_mixtures(32, max_hops * Hn, 4322)).to(dev).view(32, max_hops, Hn)

    lv_o = C.c_void_p()
    if a.out_rate != FS:
        _lib.check(h.ptr, lib.septfa_live_create_rates(h.ptr, n, W, H, a.rate, a.out_rate, C.byref(lv_o)))
        out_delay = C.c_int()
        Ho = lib.septfa_live_output_hop(lv_o, C.byref(out_delay))
        ws_o = torch.empty(lib.septfa_live_workspace_bytes(lv_o, n), dtype=torch.uint8, device=dev)
        out_o = torch.empty((n, 2, Ho), device=dev)

    st = C.c_void_p()
    _lib.check(h.ptr, lib.septfa_online_create_win(h.ptr, n, W, H, C.byref(st)))
    ws_on = torch.empty(lib.septfa_online_workspace_bytes(st), dtype=torch.uint8, device=dev)
    win = torch.from_numpy(np.tile(synth.make_mixtures(16, W, 4321), ((n + 15) // 16, 1))[:n]).to(dev)
    emitted = torch.empty((n, 2, H), device=dev)
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
    push_r_ms, launches_r = [], 0
    push_o_ms, launches_o = [], 0
    for t in range(a.warmup + a.steps):
        length = np.round((3 + (np.arange(n) + gen) % 8) * c).astype(np.int64)
        ended = np.nonzero((k == length) & (start <= t))[0].astype(np.int32)
        if ended.size:
            _lib.check(h.ptr, lib.septfa_live_release(lv, ended.ctypes.data_as(C.c_void_p), ended.size, stream))
            for other in (lv_r, lv_o):
                if other:
                    _lib.check(h.ptr, lib.septfa_live_release(other, ended.ctypes.data_as(C.c_void_p), ended.size, stream))
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
        if lv_r:
            hops_r = mixes_r[mix, torch.from_numpy(k[slots]).to(dev)].contiguous()

            def push_r():
                _lib.check(h.ptr, lib.septfa_live_push(lv_r, sl, slots.size, C.c_void_p(hops_r.data_ptr()), C.byref(ikw),
                                                       C.c_void_p(out.data_ptr()), C.c_void_p(vad.data_ptr()),
                                                       C.c_void_p(perm.data_ptr()), C.c_void_p(ws_r.data_ptr()), ws_r.numel(),
                                                       stream))
            tr = timed(push_r)
            launches_r = lib.septfa_last_launch_count(h.ptr)
        if lv_o:
            hops_o = hops_r if lv_r else hops

            def push_o():
                _lib.check(h.ptr, lib.septfa_live_push(lv_o, sl, slots.size, C.c_void_p(hops_o.data_ptr()), C.byref(ikw),
                                                       C.c_void_p(out_o.data_ptr()), C.c_void_p(vad.data_ptr()),
                                                       C.c_void_p(perm.data_ptr()), C.c_void_p(ws_o.data_ptr()), ws_o.numel(),
                                                       stream))
            to = timed(push_o)
            launches_o = lib.septfa_last_launch_count(h.ptr)
        ts = timed(step)
        k[slots] += 1
        if t >= a.warmup:
            assert slots.size == n, "timed steps must push every slot"
            push_ms.append(tp)
            if lv_r:
                push_r_ms.append(tr)
            if lv_o:
                push_o_ms.append(to)
            step_ms.append(ts)
            ns.append(int(slots.size))
            restarts.append(int(ended.size))
    lib.septfa_live_destroy(lv)
    for other in (lv_r, lv_o):
        if other:
            lib.septfa_live_destroy(other)
    lib.septfa_online_destroy(st)

    p50p, p50s, p99p = pct(push_ms, 0.5), pct(step_ms, 0.5), pct(push_ms, 0.99)
    rec = {"bench": "live_push_vs_lockstep_online_step", **gpu_info(0),
           "config": "config_with_vad, seeded weights, filter_signals_by_smo_vad",
           "window": W, "hop": H, "frames": _lib.num_frames(W), "vad_frames_per_push": n_vad,
           "streams": n, "timed_steps": len(push_ms), "warmup_steps": a.warmup,
           "stream_hops": [int(round(3 * c)), max_hops], "start_period_steps": period,
           "releases_per_step_mean": float(np.mean(restarts)),
           "push": {"p50_ms": p50p, "p99_ms": p99p, "min_ms": min(push_ms), "launches": launches},
           "lockstep_step": {"p50_ms": p50s, "p99_ms": pct(step_ms, 0.99), "min_ms": min(step_ms)},
           "push_over_step_p50": p50p / p50s,
           "realtime_streams_at_push_p99": n * (H / FS) / (p99p / 1000.0),
           "timing": "CUDA events around one call between device synchronisations; legs alternate step by step",
           "state_bytes_per_slot": 4 + 12 * (W - H)}
    if lv_r:
        p50r, p99r = pct(push_r_ms, 0.5), pct(push_r_ms, 0.99)
        rec["rate_leg"] = {"rate": a.rate, "input_hop": Hn, "delay_samples": delay.value,
                           "push": {"p50_ms": p50r, "p99_ms": p99r, "min_ms": min(push_r_ms), "launches": launches_r},
                           "overhead_p50_ms": p50r - p50p, "overhead_p99_ms": p99r - p99p,
                           "realtime_streams_at_push_p99": n * (H / FS) / (p99r / 1000.0)}
    if lv_o:
        p50o, p99o = pct(push_o_ms, 0.5), pct(push_o_ms, 0.99)
        b50, b99 = (p50r, p99r) if lv_r else (p50p, p99p)
        rec["out_rate_leg"] = {"rate": a.rate, "out_rate": a.out_rate, "output_hop": Ho, "out_delay_samples": out_delay.value,
                               "push": {"p50_ms": p50o, "p99_ms": p99o, "min_ms": min(push_o_ms), "launches": launches_o},
                               "same_session_16k_out": {"p50_ms": b50, "p99_ms": b99},
                               "overhead_p50_ms": p50o - b50, "overhead_p99_ms": p99o - b99,
                               "realtime_streams_at_push_p99": n * (H / FS) / (p99o / 1000.0)}
    line = json.dumps(rec)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
