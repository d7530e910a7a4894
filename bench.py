#!/usr/bin/env python
"""Benchmark of the Sep-TFAnet-VAD inference forward pass (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference on the host cores
    python bench.py ... --dump-outputs DIR                   # also save what the last timed step returned, to compare builds

A "step" is one forward pass over one batch of synthetic noisy two-speaker mixtures
(BASELINE.json configs[1]: config_with_vad.json, 256 x 4 s per GPU, filter_signals_by_smo_vad).
Metric: mixture-seconds processed per second, whole job (all N GPUs). Weak scaling: every rank
runs the same per-GPU batch on its own shard of mixtures; there is no collective on the data
path, torch.distributed only takes the MAX of the per-rank times.

Prints ONE JSON line (rank 0) with the keys the driver contract asks for, plus:
  roofline       - dominant kernel (tcgen05 dconv+res_out GEMM): algorithmic FLOP per launch divided by
                   its CUDA-event duration, against the measured bf16 peak (MEASURED_PEAKS.json)
  kernels        - per-kernel-class device time per step (CUDA events on the launch stream)
  e2e            - the same metric through the host API: pinned host buffers, H2D and D2H inside the timing;
                   e2e.pcie measures the plain pinned-copy ceiling of the same bytes on this box
  e2e_16bit      - the host API with int16 PCM input (normalised on the device) and fp16 output (`-ps 16`)
  cfg4 / cfg5    - BASELINE.json configs[3] (60 s, config_without_vad) and configs[4] (8192 x 4 s, sharded)
  torch_eager_b200 - the unmodified reference module moved `.to("cuda")` under stock torch eager (the stronger baseline)
  cpu_baseline   - the unmodified reference timed on this box's host cores (bounded sample)
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS = 16000
MAC_PER_FRAME = 4899657                     # SURVEY.md section 8(a): algorithmic MACs per STFT frame
DCONV_MAC_PER_FRAME = 131072 + 1536         # res_out 512->256 + depthwise k3 (the dominant kernel's share)
CONV1_MAC_PER_FRAME = 65536
NCU_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r2_dominant_traffic.json")   # {"kernel": ..., "dram_bytes_per_launch": ...}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), float(p["hbm_gbs"]), "measured"
    except Exception:  # noqa: BLE001
        return 1400.0, 6650.0, "fallback"  # /opt/skills/guides/B200_PROFILING.md


def workload_config(a):
    """The `config` object: identical for our arm and the reference arm (same workload, same inputs, same weights)."""
    return {"workload": f"config_with_vad, {a.batch} x {a.length / FS:g} s mixtures per GPU, filter_signals_by_smo_vad "
                        "(BASELINE.json configs[1])",
            "weights": "seeded random-init, reference layout (the shipped checkpoints are absent)",
            "inputs": "32 distinct seeded synthetic two-speaker mixtures per GPU, tiled to the batch",
            "l2": "working set ~0.6 GB per step >> 126 MB L2 (no explicit flush)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [v.strip() for v in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            load = [s for s in sm if s >= 0.5 * max(sm)] or sm
            out = {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def hbm_kernels(kernels, M, B, L, peak_hbm, exports):
    """Achieved HBM bandwidth of the bandwidth-class kernels: ALGORITHMIC bytes per step (compulsory traffic of the
    layout in DESIGN.md section 2, stated per frame in DESIGN.md section 3) over the class's CUDA-event time."""
    spec = 257 * 8 * M          # complex64 spectrogram
    lg = 2 * 257 * 4 * M        # both speakers' mask logits
    alg = {
        # resid: read stream fp32 + accumulators fp16, write stream fp32 (24 launches)
        "resid": 24 * M * (1024 + 512 + 1024),
        # frontend: read x, write S and the gated dB stream (+ the optional spectrum export: read stream, write [B,257,T])
        "frontend": B * L * 4 + spec + M * 1024 + ((M * 1024 + 257 * 4 * M) if exports else 0),
        # istft: read logits, S and gate, write both waveforms
        "istft": lg + spec + 2 * M * 4 + 2 * B * L * 4,
        # export: read logits and S, write est (complex64), masks and logits in torch layout
        "export": (lg + spec + 2 * spec + lg + lg) if exports else 0,
    }
    out = {}
    for k, nbytes in alg.items():
        ms = kernels.get(k, {}).get("ms_per_step", 0.0)
        if ms <= 0 or nbytes == 0:
            continue
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[k] = {"alg_bytes_per_step": int(nbytes), "ms_per_step": ms, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak_hbm}
    return out


# --------------------------------------------------------------------------- the reference on the host cores
def _all_host_threads():
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        pass
    return n


class ReferenceCPU:
    """The unmodified reference `SeparationModel` (oracle/ref_loader.py: /root/reference here, its byte-compiled copy under
    oracle/_ref on the GPU box) on the host cores, through its stock forward. Falls back to the numpy port of the oracle
    (labelled "port") only if the reference cannot be imported at all."""

    def __init__(self, length, chunk):
        import numpy as np
        from septfa_b200 import synth
        self.np, self.synth, self.length, self.chunk = np, synth, length, chunk
        self.args = synth.CONFIG_WITH_VAD
        self.kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
        self.cores = _all_host_threads()
        self.kind, self.why_port = "reference", None
        try:
            import torch
            from oracle import ref_loader
            ns = ref_loader.load()
            torch.set_num_threads(self.cores)
            warnings.filterwarnings("ignore")
            with contextlib.redirect_stdout(io.StringIO()):
                m = ns.model.SeparationModel(**self.args)
            m.load_state_dict(synth.make_state_dict(self.args, 0), strict=True)
            self.model = m.eval()
            self.torch = torch
            self.desc = (f"unmodified reference model/model.py:402-461 ({ns.kind} import), torch {torch.__version__} CPU, "
                         f"{self.cores} threads, forwards of {chunk} mixtures (its fastest CPU batch size)")
        except Exception as e:  # noqa: BLE001
            self.kind, self.why_port = "port", f"{type(e).__name__}: {e}"
            from oracle import septfa_oracle as O
            try:
                from threadpoolctl import threadpool_limits
                threadpool_limits(self.cores)
            except Exception:  # noqa: BLE001
                pass
            self.O = O
            self.W = O.OracleWeights(synth.make_state_dict_numpy(self.args, 0), self.args, np.float32)
            self.desc = f"numpy fp32 port (oracle/septfa_oracle.py; reference import failed: {self.why_port})"

    def mixtures(self, n):
        base = self.synth.make_mixtures(min(n, 32), self.length, 1234)
        return self.np.tile(base, ((n + len(base) - 1) // len(base), 1))[:n]

    def run(self, x):
        """One pass over x [n, L] in chunks; returns seconds."""
        t0 = time.perf_counter()
        for i in range(0, len(x), self.chunk):
            xb = x[i:i + self.chunk]
            if self.kind == "reference":
                with self.torch.no_grad():
                    self.model(self.torch.from_numpy(xb), dict(self.kw))
            else:
                self.O.forward(xb, self.W, dict(self.kw))
        return time.perf_counter() - t0


def run_reference(a, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    ref = ReferenceCPU(a.length, a.ref_chunk)
    # one step = the whole per-GPU workload (a.batch mixtures) unless that cannot finish in a few minutes on this host
    probe = ref.mixtures(min(a.ref_chunk, a.batch))
    ref.run(probe[:2])
    t_probe = ref.run(probe)
    per_mix = t_probe / len(probe)
    n_mix = a.ref_sample if a.ref_sample > 0 else a.batch
    budget = 200.0
    if per_mix * n_mix * (a.steps + a.warmup) > budget:
        n_mix = max(a.ref_chunk, int(budget / (per_mix * (a.steps + a.warmup))) // a.ref_chunk * a.ref_chunk)
    x = ref.mixtures(n_mix)
    for _ in range(a.warmup):
        ref.run(x)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        ref.run(x)
    dt = time.perf_counter() - t0
    value = a.steps * n_mix * a.length / FS / dt
    sample = (f"{n_mix} of the step's {a.batch} x {a.length / FS:g} s mixtures per step, {a.steps} steps; {ref.desc}")
    line = {
        "impl": "reference", "metric": "mixture-seconds processed per second (offline forward)", "value": value,
        "unit": "audio-s/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(a),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": ref.cores, "kind": ref.kind, "sample": sample},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def torch_eager_b200(a, dev, x_dev):
    """The stronger baseline (SURVEY.md section 2.2): the unmodified reference module moved `.to("cuda")`, stock torch
    eager (cuFFT + cuDNN/cuBLAS + ATen), same weights and batch. `inference_kw={}`: the gating tail of
    model/model.py:445-448 builds its smoothing conv on the CPU and raises on CUDA inputs."""
    import torch
    from septfa_b200 import synth
    try:
        from oracle import ref_loader
        ns = ref_loader.load()
        warnings.filterwarnings("ignore")
        with contextlib.redirect_stdout(io.StringIO()):
            m = ns.model.SeparationModel(**synth.CONFIG_WITH_VAD)
        m.load_state_dict(synth.make_state_dict(synth.CONFIG_WITH_VAD, 0), strict=True)
        m = m.eval().to(dev)
        with torch.no_grad():
            for _ in range(2):
                m(x_dev, {})
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = 5
            e0.record()
            for _ in range(n):
                out = m(x_dev, {})
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        B, L = x_dev.shape
        res = {"value": B * L / FS / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms, "steps": n,
               "what": f"unmodified reference SeparationModel.to('cuda') ({ns.kind} import), torch {torch.__version__} eager fp32 "
                       "(TF32 off), inference_kw={} (its gating tail raises on CUDA), inputs resident, CUDA events",
               "same_batch": [int(B), int(L)]}
        del m, out
        torch.cuda.empty_cache()
        return res
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}


def pcie_ceiling(torch, dev, h2d_bytes, d2h_bytes, reps=10):
    """Plain pinned-memory copies of one step's bytes, both directions at once on two streams: the PCIe ceiling of the
    end-to-end number on this box (and, under torchrun, with all ranks copying at the same time)."""
    src = torch.empty(h2d_bytes, dtype=torch.uint8, pin_memory=True)
    dst = torch.empty(d2h_bytes, dtype=torch.uint8, pin_memory=True)
    d_in = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
    d_out = torch.empty(d2h_bytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def go(n):
        for _ in range(n):
            with torch.cuda.stream(s1):
                d_in.copy_(src, non_blocking=True)
            with torch.cuda.stream(s2):
                dst.copy_(d_out, non_blocking=True)
        s1.synchronize()
        s2.synchronize()

    go(2)
    t0 = time.perf_counter()
    go(reps)
    dt = (time.perf_counter() - t0) / reps
    return dt


DUMP_BYTES = 60_000_000   # array data of --dump-outputs: with the .npy headers, under 64 MB in all


def dump_outputs(out_dir, returned):
    """Write the tensors a forward returned as float32 ``out_dir/<name>.npy`` (complex ones with a trailing (real, imag)
    axis). If together they exceed DUMP_BYTES, every array keeps the same batch rows: a sample drawn with a fixed seed,
    so that two runs with the same arguments write the same rows."""
    import numpy as np
    import torch
    arrays = {k: torch.view_as_real(v) if v.is_complex() else v for k, v in returned.items() if torch.is_tensor(v)}
    B = next(iter(arrays.values())).shape[0]
    row_bytes = sum(v[0].numel() * 4 for v in arrays.values())
    rows = np.arange(B)
    if B * row_bytes > DUMP_BYTES:
        if row_bytes > DUMP_BYTES:
            raise SystemExit(f"--dump-outputs: one batch row of the outputs alone is {row_bytes} bytes")
        rows = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v[torch.from_numpy(rows).to(v.device)].float().cpu().numpy())
    print(f"bench.py: wrote {', '.join(arrays)} of batch rows {rows.tolist()} to {out_dir}", file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="mixtures per GPU per step")
    ap.add_argument("--length", type=int, default=64000, help="samples per mixture (4 s @ 16 kHz)")
    ap.add_argument("--ref-sample", type=int, default=0, help="mixtures per step of the reference arm (0 = the whole batch)")
    ap.add_argument("--ref-chunk", type=int, default=64, help="mixtures per reference forward on the CPU")
    ap.add_argument("--cpu-sample", type=int, default=256, help="mixtures of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip cfg4 / cfg5 / torch-eager / 16-bit legs")
    ap.add_argument("--lean", action="store_true", help="skip the optional exports (est/mask/spectrum/logits)")
    ap.add_argument("--online-streams", type=int, default=1024, help="concurrent streams of the online leg (0 = skip)")
    ap.add_argument("--online-hops", type=int, default=12)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed forward returned (rank 0) as DIR/<name>.npy, "
                         "float32; a fixed, seeded sample of the batch rows when all of it would exceed 64 MB")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; it cannot be combined with --impl reference")

    # NCCL logs (its version banner included, which WARN and VERSION both print) go to stdout by default and would
    # precede the JSON line: send them to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[v] = str(_all_host_threads())  # torchrun forces OMP_NUM_THREADS=1
        run_reference(a, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from septfa_b200 import synth
    from septfa_b200.model import SeparationModel
    from septfa_b200.shard import gather_max_time, shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    args = synth.CONFIG_WITH_VAD
    with contextlib.redirect_stdout(io.StringIO()):
        model = SeparationModel(**args)
    model.load_state_dict(synth.make_state_dict(args, 0), strict=True)
    model.eval().to(dev)
    if a.lean:
        model.materialize.update(estimated_stfts=False, mask_per_speaker=False, spectrum=False, masks_b=False)
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)

    # this rank's shard of the global batch (distinct mixtures per rank; 32 distinct ones tiled)
    B, L = a.batch, a.length
    g0, _ = shard_range(world * B, rank, world)
    n_distinct = min(B, 32)
    base = synth.make_mixtures(n_distinct, L, 1234, first_index=g0)
    x_host = torch.from_numpy(np.tile(base, ((B + n_distinct - 1) // n_distinct, 1))[:B]).pin_memory()
    x_dev = x_host.to(dev)
    T = 1 + L // 256

    def step():
        return model(x_dev, kw)

    for _ in range(max(a.warmup, 3)):
        step()
    torch.cuda.synchronize()

    # ---- device-resident throughput (`value`): CUDA events on the launch stream, max over ranks
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for _ in range(a.steps):
        last = None       # release the previous step's outputs before the next forward allocates its own
        last = step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_dev = gather_max_time(e0.elapsed_time(e1) * 1e-3)
    launches = model.last_launch_count * a.steps
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, dict(zip(("out", "output_vad", "estimated_stfts"), last)))
    del last

    # ---- per-kernel-class timing (separate pass; events inside forward on the same stream)
    model.set_profile(True)
    for _ in range(a.steps):
        step()
    prof = model.read_profile(dev)
    model.set_profile(False)
    kernels = {k: {"ms_per_step": v[0] / a.steps, "launches_per_step": v[1] / a.steps} for k, v in prof.items()}

    # ---- end to end through the public host API (pinned host buffers, H2D + D2H inside)
    out_h = None
    for _ in range(2):
        out_h = model.forward_host(x_host, kw, device=local_rank)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        out_h = model.forward_host(x_host, kw, device=local_rank)
    t_e2e_sync = gather_max_time(time.perf_counter() - t0)
    assert out_h[0].shape == (B, 2, L)

    # ---- the same through the batch-stream API (forward_host_submit / result, three slots in rotation): every step still copies
    # its input from pinned host memory and its results back to pinned host memory; successive steps overlap their
    # PCIe copies with each other's kernels, which is how a file loop (only_inference.py:80-100) would call it.
    # The timed region runs from the first submit to the last result (pipeline fill and drain included).
    def stream_leg(xs, out_dtype):
        NS = 3   # pipeline slots in rotation: with two, the copy-in of step i + 1 queues behind the copy-out of step i - 1
        outs = [torch.empty((B, 2, L), dtype=out_dtype, pin_memory=True) for _ in range(NS)]
        vads = [torch.empty((B, 2, T), dtype=torch.float32, pin_memory=True) for _ in range(NS)]

        def stream_steps(n):
            pend = [None] * NS
            for i in range(n):
                sl = i % NS
                if pend[sl] is not None:
                    pend[sl].result()
                pend[sl] = model.forward_host_submit(xs[i & 1], kw, device=local_rank, slot=sl, out=outs[sl], vad=vads[sl],
                                                     out_dtype=out_dtype)
            for f in pend:
                if f is not None:
                    f.result()

        stream_steps(4)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        stream_steps(a.steps)
        return gather_max_time(time.perf_counter() - t0), outs, vads

    t_e2e, outs, _ = stream_leg([x_host, x_host.clone().pin_memory()], torch.float32)
    # same results as the synchronous call up to the fp16 operand noise: the two paths tile the batch differently, so a
    # VAD probability within ~4e-4 of the threshold may flip a frame's gate (allowed: |p - thr| < 1e-3) in a few clips
    assert torch.isfinite(outs[0]).all()
    assert ((outs[0] - out_h[0]).abs().amax(dim=(1, 2)) > 1e-3).float().mean().item() < 0.1
    h2d_bytes, d2h_bytes = int(x_host.numel() * 4), int(B * 2 * L * 4 + B * 2 * T * 4)
    t_pcie = gather_max_time(pcie_ceiling(torch, dev, h2d_bytes, d2h_bytes))

    # ---- 16-bit host formats: int16 PCM in (as a wav file holds it; converted and min-max normalised on the device,
    # only_inference.py:69,81) and fp16 out (save_audio's `-ps 16`, utlis_inference.py:30-32): half the PCIe bytes
    e2e16 = None
    if not a.no_extras:
        pcm = torch.from_numpy(np.round(x_host.numpy() / 0.9 * 32767.0).astype(np.int16)).pin_memory()
        t16, outs16, _ = stream_leg([pcm, pcm.clone().pin_memory()], torch.float16)
        assert torch.isfinite(outs16[0].float()).all()
        t_pcie16 = gather_max_time(pcie_ceiling(torch, dev, h2d_bytes // 2, B * 2 * L * 2 + B * 2 * T * 4))
        e2e16 = {"t": t16, "t_pcie": t_pcie16}
        del outs16
    clocks = sampler.stop() if sampler else None   # sampled over the timed, profiled and end-to-end legs

    # ---- online mode (BASELINE.json configs[2]): S concurrent streams, one hop-step = forward on the current 3 s
    # windows + per-stream L1-PIT + reorder + append; latency per hop-step from CUDA events, windows resident
    online = None
    if a.online_streams > 0 and rank == 0:
        import ctypes as C
        from septfa_b200 import lib as _lib
        S = a.online_streams
        h = model._handle(dev)
        st = C.c_void_p()
        _lib.check(h.ptr, h.lib.septfa_online_create(h.ptr, S, C.byref(st)))
        ws = torch.empty(h.lib.septfa_online_workspace_bytes(st), dtype=torch.uint8, device=dev)
        win = torch.from_numpy(np.tile(synth.make_mixtures(16, 48000, 4321), ((S + 15) // 16, 1))[:S]).to(dev)
        emitted = torch.empty((S, 2, 16000), dtype=torch.float32, device=dev)
        perm = torch.empty((S, 2), dtype=torch.int32, device=dev)
        ikw = _lib.InferKw.from_dict(kw)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        times = []
        for i in range(a.online_hops + 3):
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            _lib.check(h.ptr, h.lib.septfa_online_step(st, C.c_void_p(win.data_ptr()), C.byref(ikw), C.c_void_p(emitted.data_ptr()),
                                                       C.c_void_p(perm.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(), stream))
            s1.record()
            torch.cuda.synchronize()
            if i >= 3:
                times.append(s0.elapsed_time(s1))
        h.lib.septfa_online_destroy(st)
        del ws
        times.sort()
        p50 = times[len(times) // 2]
        p99 = times[min(len(times) - 1, int(0.99 * len(times)))]
        online = {"streams": S, "hops_timed": len(times), "p50_ms_per_hop_step": p50, "p99_ms_per_hop_step": p99,
                  "p50_ms_per_frame": p50 / 62.5, "p99_ms_per_frame": p99 / 62.5,
                  "audio_s_per_s": S * 1.0 / (p50 * 1e-3),
                  "note": "hop-step = forward on S x 3 s windows (T=188) + per-stream L1-PIT + reorder + emit 1 s; "
                          "ms per frame = hop-step / 62.5 frames per hop (the reference has no per-frame entry point)"}

    # ---- BASELINE.json configs[4]: 8192 x 4 s with the VAD gate, sharded over the ranks, streamed in 256-mixture host
    # batches through forward_host_stream (host input and output every batch); whole-job audio-s/s, max over ranks
    cfg5 = None
    if not a.no_extras:
        total = 8192
        n_mine = shard_range(total, rank, world)[1] - shard_range(total, rank, world)[0]
        nb = n_mine // B
        xs = [x_host, x_host.clone().pin_memory()]
        for _ in model.forward_host_stream((xs[i & 1] for i in range(6)), kw, device=local_rank, reuse_outputs=True):
            pass
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        n_out = 0
        for o, v in model.forward_host_stream((xs[i & 1] for i in range(nb)), kw, device=local_rank, reuse_outputs=True):
            n_out += o.shape[0]
        t5 = gather_max_time(time.perf_counter() - t0)
        assert n_out == nb * B
        cfg5 = {"workload": f"{total} x 4 s mixtures over {world} GPU(s) in host batches of {B} (BASELINE.json configs[4])",
                "value": world * nb * B * L / FS / t5, "unit": "audio-s/s", "seconds": t5,
                "api": "SeparationModel.forward_host_stream(reuse_outputs=True): float32 pinned host input and output per batch"}

    # ---- BASELINE.json configs[3]: 60 s mixtures, config_without_vad (stresses the per-utterance global statistics)
    cfg4 = None
    if not a.no_extras and rank == 0:
        with contextlib.redirect_stdout(io.StringIO()):
            m4 = SeparationModel(**synth.CONFIG_WITHOUT_VAD)
        m4.load_state_dict(synth.make_state_dict(synth.CONFIG_WITHOUT_VAD, 0), strict=True)
        m4.eval().to(dev)
        m4.materialize.update(estimated_stfts=False, mask_per_speaker=False, spectrum=False, masks_b=False)
        cfg4 = {"workload": "config_without_vad, 60 s mixtures, inference_kw={} (BASELINE.json configs[3])", "unit": "audio-s/s"}
        x60 = torch.from_numpy(np.tile(synth.make_mixtures(4, 960000, 777), (8, 1))).to(dev)
        for nb4 in (1, 32):
            xb = x60[:nb4]
            for _ in range(3):
                m4(xb, {})
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(5):
                m4(xb, {})
            s1.record()
            torch.cuda.synchronize()
            ms = s0.elapsed_time(s1) / 5
            cfg4[f"batch_{nb4}"] = {"ms_per_forward": ms, "value": nb4 * 60.0 / (ms * 1e-3),
                                    "mfu": 2.0 * MAC_PER_FRAME * nb4 * 3751 / (ms * 1e-3) / 1e12 / measured_peaks()[0]}
        del m4, x60
        torch.cuda.empty_cache()

    eager = None
    if not a.no_extras and rank == 0:
        eager = torch_eager_b200(a, dev, x_dev)

    # ---- small-request latency (SURVEY.md section 8(f) rank 4): one 4 s mixture, resident input, per-call CUDA events;
    # the eager launch sequence (~80 kernels) against its CUDA-graph replay (SeparationModel.graphed)
    small = None
    if not a.no_extras and rank == 0:
        def lat(fn, n=200):
            for _ in range(10):
                fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(n):
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                fn()
                s1.record()
                s1.synchronize()
                ts.append(s0.elapsed_time(s1))
            ts.sort()
            return {"p50_ms": ts[len(ts) // 2], "p99_ms": ts[min(len(ts) - 1, int(0.99 * len(ts)))]}
        model.materialize.update(estimated_stfts=False, mask_per_speaker=False, spectrum=False, masks_b=False)
        x1 = x_dev[:1].contiguous()
        small = {"workload": "one 4 s mixture per request, input resident, VAD gate on", "eager": lat(lambda: model(x1, kw))}
        try:
            g1 = model.graphed(1, L, kw)
            g1.x.copy_(x1)
            small["cuda_graph"] = dict(lat(g1.replay), nodes=g1.num_nodes)
        except Exception as e:  # noqa: BLE001
            small["cuda_graph"] = {"unavailable": f"{type(e).__name__}: {e}"}
        if not a.lean:
            model.materialize.update(estimated_stfts=True, mask_per_speaker=True, spectrum=True, masks_b=True)

    if rank == 0:
        audio_s = world * B * L / FS * a.steps
        peak_tf, peak_hbm, peak_src = measured_peaks()
        M = B * T
        d_ms, d_n = prof["dconv"]
        dconv_ms = d_ms / max(d_n, 1)
        flop_per_launch = 2.0 * DCONV_MAC_PER_FRAME * M
        achieved = flop_per_launch / (dconv_ms * 1e-3) / 1e12 if dconv_ms > 0 else 0.0
        c_ms, c_n = prof["conv1"]
        conv1_tf = 2.0 * CONV1_MAC_PER_FRAME * M / (c_ms / max(c_n, 1) * 1e-3) / 1e12 if c_ms > 0 else 0.0
        traffic, traffic_src = None, None
        try:
            with open(NCU_TRAFFIC_FILE) as f:
                tj = json.load(f)
            if (B, L) == (256, 64000):
                traffic, traffic_src = tj["dram_bytes_per_launch"], tj.get("source")
        except Exception:  # noqa: BLE001
            pass
        cfg = workload_config(a)
        line = {
            "metric": "mixture-seconds processed per second (offline forward)",
            "value": audio_s / t_dev, "unit": "audio-s/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": 1e3 * t_dev / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16xf16->f32 (tcgen05), f32 elsewhere", "data": "synthetic",
            "config": cfg,
            "frames_per_step_per_gpu": M, "exports": not a.lean,
            "model_flops_utilization": 2.0 * MAC_PER_FRAME * M * world * a.steps / t_dev / 1e12 / (peak_tf * world),
            "roofline": {"kernel": "dconv + res_out (depthwise dilated conv -> PReLU -> 512->256 tcgen05 GEMM, model.py:136-144)",
                         "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved / peak_tf, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "ms_per_launch": dconv_ms, "flop_per_launch": flop_per_launch,
                         "conv1_tflops": conv1_tf},
            "kernels": kernels,
            "hbm_kernels": hbm_kernels(kernels, M, B, L, peak_hbm, not a.lean),
            "e2e": {"value": audio_s / t_e2e, "unit": "audio-s/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "ms_per_step": 1e3 * t_e2e / a.steps,
                    "pcie": {"ms_per_step_copies_only": 1e3 * t_pcie,
                             "pcie_gbs": (h2d_bytes + d2h_bytes) / t_pcie / 1e9,
                             "frac_of_pcie": t_pcie / (t_e2e / a.steps),
                             "what": "pinned H2D and D2H copies of one step's bytes, both directions at once, all ranks at the "
                                     "same time, no kernels: the copy-only floor of a step on this box"},
                    "api": "SeparationModel.forward_host_submit / HostBatch.result (septfa_forward_host_submit_fmt / _wait), "
                           "three batches in flight (pipeline slots in rotation); pinned host input and output per step; fill and drain inside the timing"},
            "e2e_sync": {"value": audio_s / t_e2e_sync, "unit": "audio-s/s", "ms_per_step": 1e3 * t_e2e_sync / a.steps,
                         "api": "SeparationModel.forward_host (septfa_forward_host): one synchronous call per step, "
                                "two-chunk copy/compute pipeline inside the call"},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        if e2e16 is not None:
            line["e2e_16bit"] = {"value": audio_s / e2e16["t"], "unit": "audio-s/s", "ms_per_step": 1e3 * e2e16["t"] / a.steps,
                                 "h2d_bytes_per_step": h2d_bytes // 2, "d2h_bytes_per_step": int(B * 2 * L * 2 + B * 2 * T * 4),
                                 "pcie": {"ms_per_step_copies_only": 1e3 * e2e16["t_pcie"],
                                          "frac_of_pcie": e2e16["t_pcie"] / (e2e16["t"] / a.steps)},
                                 "api": "forward_host_submit with int16 PCM input (astype float32 + min-max normalise on the "
                                        "device, only_inference.py:69,81) and out_dtype=float16 (save_audio -ps 16)"}
        if online is not None:
            line["online"] = online
        if cfg4 is not None:
            line["cfg4"] = cfg4
        if cfg5 is not None:
            line["cfg5"] = cfg5
        if eager is not None:
            line["torch_eager_b200"] = eager
        if small is not None:
            line["small_request_latency"] = small
        if world == 1 and not a.no_cpu_baseline:
            ref = ReferenceCPU(L, a.ref_chunk)
            xs = ref.mixtures(a.cpu_sample)
            ref.run(xs[:2])
            secs = ref.run(xs)
            line["cpu_baseline"] = {"value": a.cpu_sample * L / FS / secs, "unit": "audio-s/s", "cores": ref.cores,
                                    "kind": ref.kind,
                                    "sample": f"{a.cpu_sample} x {L / FS:g} s mixtures, one pass ({secs:.1f} s); {ref.desc}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
