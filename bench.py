#!/usr/bin/env python
"""Benchmark of the FastDiff reverse-diffusion sampling hot path (BASELINE.json metric:
audio samples/sec (22.05 kHz) at N=4 reverse steps).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # CPU yardstick (oracle port of the reference)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's output as DIR/<name>.npy

A "step" = one complete sampling call (all N=4 reverse steps incl. noise generation) over one batch of
synthetic input.  Workload at every N: BASELINE.json configs[1] per GPU -- batch 8 x 10 s synthetic mel
(T'=861, L=220,416), LJSpeech network, random-init weights -- i.e. weak scaling, utterances sharded over
ranks, one NCCL broadcast of the packed weights at load, no per-step collective.
Prints ONE JSON line on rank 0 (stdout); everything else goes to stderr.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

N4_SCHEDULE = [3.2176e-04, 2.5743e-03, 2.5376e-02, 7.0414e-01]  # modules/FastDiff/task/FastDiff.py:88-89
FLOP_PER_SAMPLE_STEP = 222601.0      # SURVEY.md section 8(d), torch FlopCounterMode on the reference
KC_FLOP_PER_FRAME = 2.0 * 24832 * 192  # kernel_conv+bias_conv GEMM: 2*N*K per mel frame per LVC block
METRIC = "audio samples/sec (22.05 kHz) at N=4 reverse steps"
UNIT = "samples/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# stdout must carry exactly ONE JSON line.  Libraries (NCCL's version banner, the sampler's reference-compatible prints) write
# to fd 1 behind Python's back, so fd 1 is pointed at stderr for the whole run and the JSON goes to the saved descriptor.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)
sys.stdout = sys.stderr


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"tensor": float(p["bf16_tflops_sustained"]), "tensor_burst": float(p["bf16_tflops"]), "hbm": float(p["hbm_gbs"]),
                "src": "MEASURED_PEAKS.json"}
    except Exception:
        return {"tensor": 1400.0, "tensor_burst": 1590.0, "hbm": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock / power / throttle reasons sampled DURING the timed regions: NVML polled every ~5 ms from a thread that is
    started before the warm-up (so it is already running when the short timed region begins); only samples whose host
    timestamp falls inside a [mark_begin, mark_end] window are reported.  Falls back to `nvidia-smi -lms` if NVML is missing."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.rows, self.windows, self._t0 = index, [], [], None
        self._stop = threading.Event()
        self.thr = None
        self.backend = None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:
                    idx = self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = [getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)]
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons

            def poll():
                while not self._stop.is_set():
                    try:
                        t = time.perf_counter()
                        sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                        pw = nv.nvmlDeviceGetPowerUsage(h) / 1e3
                        rs = int(get_reasons(h))
                        self.rows.append((t, sm, mx, pw, [n for n, b in zip(self.NAMES, bits) if rs & b]))
                    except Exception:
                        pass
                    time.sleep(0.004)
            self.backend = "nvml"
        except Exception as e:
            log("NVML unavailable (%r); falling back to nvidia-smi" % (e,))
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            try:
                proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                        stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except Exception as e2:  # pragma: no cover
                log("clock sampler unavailable:", e2)
                return
            self.proc = proc

            def poll():
                for line in proc.stdout:
                    c = [x.strip() for x in line.split(",")]
                    try:
                        self.rows.append((time.perf_counter(), float(c[0]), float(c[1]), float(c[2]),
                                          [n for n, v in zip(self.NAMES, c[3:7]) if v.lower().startswith("active")]))
                    except Exception:
                        pass
                    if self._stop.is_set():
                        break
            self.backend = "nvidia-smi"
        self.thr = threading.Thread(target=poll, daemon=True)
        self.thr.start()

    def mark_begin(self):
        self._t0 = time.perf_counter()

    def mark_end(self):
        if self._t0 is not None:
            self.windows.append((self._t0, time.perf_counter()))
            self._t0 = None

    def stop(self):
        if self.thr is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0}
        self._stop.set()
        if getattr(self, "proc", None):
            self.proc.terminate()
        self.thr.join(timeout=2)
        rows = [r for r in self.rows if any(a <= r[0] <= b for a, b in self.windows)]
        sm = [r[1] for r in rows]
        reasons = sorted({n for r in rows for n in r[4]}, key=self.NAMES.index)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(r[2] for r in rows) if rows else None,
                "reasons": reasons, "samples": len(rows), "power_w_max": max(r[3] for r in rows) if rows else None,
                "source": f"{self.backend}, polled during the timed regions (device-resident + e2e)"}


WORKLOAD = "batch=8 x 10 s synthetic mel (T'=861) per GPU, N=4, LJSpeech config, random-init weights"


def bench_config(world):
    """The `config` object -- identical for both arms (`--impl ours` / `--impl reference`) at the same N."""
    return {"workload": WORKLOAD, "global_batch": world * 8, "frames_per_utterance": 861, "reverse_steps": 4,
            "parallelism": f"batch-shard x{world} (weights broadcast once, no per-step collective)",
            "l2": "inputs+activations per call (>=450 MB) exceed the 126 MB L2; no explicit flush"}


class CpuYardstick:
    """The reference's CPU implementation of the path on the host cores (fp32, all intra-op threads).

    kind "reference": the UNMODIFIED reference (`sampling_given_noise_schedule` over `FastDiff.forward`,
    modules/FastDiff/module/util.py:158-235) imported from the checkout named by FD_REFERENCE_ROOT or from its bytecode build
    oracle/_ref (oracle/stage_reference.py), `.cuda()` shimmed to identity.  kind "port": oracle/fastdiff_oracle.py -- only when no copy of
    the reference is reachable (it is ~3.8x slower than the reference: its LVC is three einsum taps where the reference unfolds
    once and calls bmm; say so wherever the number is shown)."""

    def __init__(self, seed=1234):
        from fastdiff_b200.synthetic import make_state_dict
        from oracle import refimport
        sd = make_state_dict(seed)
        self.kind = "reference" if refimport.reference_root() else "port"
        if self.kind == "reference":
            self.R = refimport.load("cpu")
            self.model = self.R.FastDiff().eval()
            self.model.load_state_dict(sd)
            self.dh = self.R.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
            self.where = self.R.root
        else:
            from oracle import fastdiff_oracle as O
            self.O, self.W = O, O.fold_weight_norm(sd)
            self.dh = O.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
            self.where = "oracle/fastdiff_oracle.py"

    def sample_once(self, B, Tm):
        """One complete N=4 sampling call; returns seconds."""
        from fastdiff_b200.synthetic import make_inputs
        _, mel = make_inputs(B, Tm, 0)
        sched = torch.FloatTensor(N4_SCHEDULE)
        t0 = time.perf_counter()
        with torch.no_grad(), contextlib.redirect_stdout(sys.stderr):
            if self.kind == "reference":
                self.R.sampling_given_noise_schedule(self.model, (B, 1, Tm * 256), self.dh, sched, condition=mel, ddim=False,
                                                     return_sequence=False)
            else:
                self.O.sample(self.W, (B, 1, Tm * 256), self.dh, sched, mel)
        return time.perf_counter() - t0

    def describe(self, sample):
        return {"unit": UNIT, "cores": torch.get_num_threads(), "kind": self.kind, "sample": sample, "host_cpus": os.cpu_count(),
                "source": self.where, "torch_threads": torch.get_num_threads()}


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path (see CpuYardstick), all host threads.  A step = one
    complete N=4 sampling call on a BOUNDED sample of the workload: 1 of the 8 utterances of a batch (B=1 x 10 s).  (The reference
    is FASTER per sample at B=1 than at B=8 -- SURVEY.md section 6: 74 k vs 47 k samples/s on 8 cores -- so the bounded sample
    favours the reference.)  Under torchrun only rank 0 runs; the other ranks exit 0 without work."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cy = CpuYardstick()
    B, Tm = 1, 861
    for _ in range(args.warmup):
        cy.sample_once(B, Tm)
    ts = [cy.sample_once(B, Tm) for _ in range(args.steps)]
    per = sum(ts) / len(ts)
    val = B * Tm * 256 / per
    sample = (f"{'UNMODIFIED reference' if cy.kind == 'reference' else 'oracle port of the reference'} (torch CPU fp32, "
              f"{torch.get_num_threads()} threads): 1 utterance x 10 s of the 8 x 10 s batch, all N=4 reverse steps, per step")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(world),
        "cpu_baseline": {"value": val, **cy.describe(sample)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_ours(args):
    """This repo's arm.  Every rank drives the PRODUCT multi-GPU API -- fastdiff_b200.shard.ShardedFastDiff (one NCCL broadcast of the
    packed weights at construction, then `sample()` on this rank's slice of the global batch, no per-step collective) -- also at N = 1,
    where it degenerates to one engine.  Three timed regions:
      value  device-resident: mel already in HBM, noise drawn on the device (Philox), CUDA events, max over ranks;
      e2e    the same call with HOST buffers: pinned mel -> device and waveform -> pinned host inside the timed region;
      e2e_reference_noise (N = 1)  `fastdiff_b200.sampling_given_noise_schedule` in its drop-in default `noise_mode="reference"`:
             x_T and the N-1 noise tensors are drawn on the CPU default generator in the reference's order and copied H2D
             (bit-compatible RNG stream; host RNG time inside the timed region)."""
    import torch.distributed as dist
    import fastdiff_b200 as fb
    from fastdiff_b200.shard import ShardedFastDiff
    from fastdiff_b200.synthetic import make_inputs, make_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B, Tm = args.batch, args.frames          # per GPU (weak scaling)
    L = Tm * 256
    GB = world * B

    # ---- weights: rank 0 packs, ONE broadcast of the blob (inside ShardedFastDiff), every rank loads from device memory -------
    t_load0 = time.perf_counter()
    sh = ShardedFastDiff(make_state_dict(1234) if rank == 0 else None, device=dev)
    torch.cuda.synchronize()
    load_s = time.perf_counter() - t_load0
    eng = sh.engine
    if args.mode:
        eng.set_mode(args.mode)
    for kv in args.opt:
        key, val = kv.split("=")
        eng.set_option(key, int(val))
    mode_name = {0: "fp32_simt", 1: "tc_3xtf32", 2: "tc_tf32", 3: "tc_3xf16"}[eng.get_mode()]

    dh = fb.compute_hyperparams_given_schedule(torch.linspace(1e-6, 0.01, 1000))
    sched = torch.FloatTensor(N4_SCHEDULE)
    # the global batch of mels: every rank builds the same tensor and ShardedFastDiff slices its own utterances out of it
    mel_host = torch.cat([make_inputs(B, Tm, seed=r)[1] for r in range(world)], 0)
    mel_dev = mel_host.to(dev)
    size = (GB, 1, L)

    def one_call(i):
        with contextlib.redirect_stdout(sys.stderr):
            return sh.sample(size, dh, sched, mel_dev, seed=1000 + i)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.start()
    for i in range(args.warmup):
        one_call(i)
    barrier()

    # ---- timed region 1: device-resident inputs (the library replays its captured CUDA graph of the whole call) -------------
    l0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if clocks:
        clocks.mark_begin()
    ev0.record()
    for i in range(args.steps):
        out = one_call(args.warmup + i)
    ev1.record()
    barrier()
    if clocks:
        clocks.mark_end()
    ms = ev0.elapsed_time(ev1)
    last_out = out.cpu() if args.dump_outputs else None
    launches = eng.launch_count() - l0
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = GB * L / (ms_per_step * 1e-3)

    # ---- timed region 1b: the same K calls with two CUDA events around EVERY kernel launch (on its own stream): per-kernel durations for the
    #      roofline.  Event recording forces plain launches (no graph replay), so this loop is a little slower than region 1.
    eng.set_option("overlap", 0)   # serial order: every class is timed alone (with the side stream on, the DBlock chain shares the SMs with embed / KP / GEMM)
    for i in range(2):
        one_call(i)
    eng.timing_enable(True)
    eng.timing_report()
    evi0, evi1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if clocks:
        clocks.mark_begin()
    evi0.record()
    for i in range(args.steps):
        one_call(args.warmup + args.steps + i)
    evi1.record()
    barrier()
    if clocks:
        clocks.mark_end()
    ms_instr = evi0.elapsed_time(evi1) / args.steps
    per_kernel = eng.timing_report()
    eng.timing_enable(False)
    eng.set_option("overlap", 1)
    saturated = eng.check_saturation()

    # ---- timed region 2: e2e, host buffers (H2D of the mels, D2H of the waveform inside) ------------------------------------
    def timed_host_loop(fn):
        fn(0)
        barrier()
        if clocks:
            clocks.mark_begin()
        t0 = time.perf_counter()
        for i in range(args.steps):
            fn(1 + i)
        barrier()
        dt = time.perf_counter() - t0
        if clocks:
            clocks.mark_end()
        tt = torch.tensor([dt], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    e2e = None
    e2e_ref_noise = None
    lo, hi = sh.my_slice(GB)
    try:
        mel_pinned = mel_host.pin_memory()
        out_host = torch.empty((hi - lo, 1, L), dtype=torch.float32).pin_memory()

        def e2e_call(i):
            with contextlib.redirect_stdout(sys.stderr):
                y = sh.sample(size, dh, sched, mel_pinned[lo:hi].to(dev, non_blocking=True), seed=5000 + i, presliced=True)
            out_host.copy_(y, non_blocking=True)
            torch.cuda.synchronize()
        dt = timed_host_loop(e2e_call)
        e2e = {"value": GB * L * args.steps / dt, "unit": UNIT, "h2d_bytes_per_step": GB * 80 * Tm * 4, "d2h_bytes_per_step": GB * L * 4,
               "ms_per_step": dt / args.steps * 1e3, "api": "fastdiff_b200.shard.ShardedFastDiff.sample (pinned host mel in, pinned host waveform out)",
               "noise": "device (Philox4x32-10)"}
    except Exception as e:  # pragma: no cover
        log("e2e leg failed:", repr(e))
    if world == 1:
        try:   # the drop-in default: reference RNG stream drawn on the host
            net = fb.FastDiff().to(dev).eval()
            net.load_state_dict(make_state_dict(1234))
            net.noise_mode = "reference"
            if args.mode:
                net.mode = args.mode
            eng_r = net.engine(dev)
            for kv in args.opt:
                key, val = kv.split("=")
                eng_r.set_option(key, int(val))
            n_ref = max(2, min(args.steps, 5))
            out_r = torch.empty((B, 1, L), dtype=torch.float32).pin_memory()

            def ref_call(i):
                with contextlib.redirect_stdout(sys.stderr):
                    y = fb.sampling_given_noise_schedule(net, (B, 1, L), dh, sched, condition=mel_pinned.to(dev, non_blocking=True))
                out_r.copy_(y, non_blocking=True)
                torch.cuda.synchronize()
            ref_call(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(n_ref):
                ref_call(i)
            dt = time.perf_counter() - t0
            e2e_ref_noise = {"value": B * L * n_ref / dt, "unit": UNIT, "ms_per_step": dt / n_ref * 1e3, "steps": n_ref,
                             "h2d_bytes_per_step": B * 80 * Tm * 4 + 4 * B * L * 4, "d2h_bytes_per_step": B * L * 4,
                             "api": "fastdiff_b200.sampling_given_noise_schedule, noise_mode='reference' (the drop-in default: x_T and 3 noise "
                                    "tensors drawn on the CPU default generator in the reference's order, copied H2D)",
                             "host_threads": torch.get_num_threads()}
            del net, eng_r
        except Exception as e:  # pragma: no cover
            log("e2e (reference noise) leg failed:", repr(e))

    clk = clocks.stop() if clocks else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"audio" if world == 1 else f"audio_rank{rank}": last_out}, DUMP_LIMIT_BYTES // world)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (live CUDA-event time inside the timed region) -------------------------------------
    peaks = measured_peaks()
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms"]) if per_kernel else None
    roofline = None
    frames = B * Tm
    samples = B * L
    n_rev = 4 * args.steps                                            # reverse steps inside the instrumented loop
    lvc_flop = 2.0 * 96 * 32 + 2.0 * 96 * 64                          # dilated conv + LVC per sample and layer
    flop_per_rev_step = {                                             # algorithmic FLOPs of a class per reverse step (SURVEY 8(d) breakdown)
        "kc_gemm": KC_FLOP_PER_FRAME * frames * 3,                    # one launch covers the 3 LVC blocks
        "lvc_layer_b2": 4 * lvc_flop * samples, "lvc_layer_b1": 4 * lvc_flop * samples / 4, "lvc_layer_b0": 4 * lvc_flop * samples / 32,
        "dblock": 7880.0 * samples, "upsample": 5248.0 * samples, "final_update": 448.0 * samples,
        "kp_hidden": (114072.0 - 110592.0 - 1152.0) * samples,       # kernel predictor minus kernel_conv / bias_conv
        "embed": 0.9e6 * B,
    }
    traffic_tab = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            traffic_tab = json.load(f)
    except Exception:
        pass
    class_roofline = {}
    for k, v in per_kernel.items():
        if k in flop_per_rev_step and v["ms"] > 0:
            a = flop_per_rev_step[k] * n_rev / (v["ms"] * 1e-3) / 1e12
            class_roofline[k] = {"tflops": a, "frac": a / peaks["tensor"], "launches_per_reverse_step": v["n"] / n_rev,
                                 "ms_per_reverse_step": v["ms"] / n_rev}
    if dom and dom in flop_per_rev_step:
        n_dom = per_kernel[dom]["n"]
        avg_ms = per_kernel[dom]["ms"] / n_dom
        flop_per_launch = flop_per_rev_step[dom] * n_rev / n_dom
        ach = flop_per_launch / (avg_ms * 1e-3) / 1e12
        tr = traffic_tab.get(dom) if (B, Tm) == (8, 861) else None
        roofline = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peaks["tensor"], "unit": "TFLOP/s",
                    "frac": ach / peaks["tensor"], "traffic": tr["dram_bytes_per_launch"] if tr else None,
                    "traffic_note": ({"source": tr["source"], "layout_minimum_bytes_per_launch": tr.get("layout_minimum_bytes_per_launch"),
                                      "what": "dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu --set full); layout_minimum = the bytes this "
                                              "kernel's data layout must move (rows in + rows out + predicted kernels), NOT SURVEY 8(d)'s algorithmic bytes"}
                                     if tr else None),
                    "peak_source": peaks["src"] + " bf16_tflops_sustained (of measured)",
                    "avg_launch_ms": avg_ms, "launches": n_dom, "share_of_step": per_kernel[dom]["ms"] / (ms_instr * args.steps),
                    "algorithmic_flop_per_launch": flop_per_launch, "mode": mode_name,
                    "timed": "CUDA events around every launch of the class on its own stream, serial kernel order (side stream off), inside bench.py",
                    "note": "fp32-level mode: every algorithmic FLOP costs 3 fp16 MMAs, so this kernel's own tensor ceiling is 1/3 of the bf16 peak"}
    step_alg_bytes = samples * 12 + frames * 320 + 61e6   # SURVEY 8(d): x in/out + z per sample, mel, folded fp32 weights once per reverse step
    whole = {"achieved_tflops": FLOP_PER_SAMPLE_STEP * 4 * GB * L / (ms_per_step * 1e-3) / 1e12,
             "frac_of_bf16_sustained": FLOP_PER_SAMPLE_STEP * 4 * B * L / (ms_per_step * 1e-3) / 1e12 / peaks["tensor"],
             "algorithmic_bytes_per_reverse_step": step_alg_bytes,
             "dram_bytes_per_reverse_step": traffic_tab.get("_per_reverse_step", {}).get("dram_bytes") if (B, Tm) == (8, 861) else None,
             "dram_bytes_source": traffic_tab.get("_per_reverse_step", {}).get("source") if (B, Tm) == (8, 861) else None}

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only) ----------------------------------------------------------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu:
        try:
            cy = CpuYardstick()
            cy.sample_once(1, 86)  # warm-up (1 s)
            reps = [cy.sample_once(1, 861) for _ in range(3 if cy.kind == "reference" else 1)]
            tcpu = min(reps)
            cpu_baseline = {"value": 861 * 256 / tcpu, **cy.describe(
                f"{'UNMODIFIED reference' if cy.kind == 'reference' else 'oracle port of the reference'} (torch CPU fp32): 1 utterance x 10 s "
                f"of the batch, all N=4 steps, best of {len(reps)} runs"), "seconds": tcpu}
        except Exception as e:  # pragma: no cover
            log("cpu baseline failed:", repr(e))

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if mode_name != "tc_tf32" else "tf32", "data": "synthetic",
        "config": (bench_config(world) if (B, Tm) == (8, 861) else
                   {**bench_config(world), "workload": f"batch={B} x {Tm * 256 / 22050:.1f} s synthetic mel (T'={Tm}) per GPU, N=4, LJSpeech config, "
                    "random-init weights", "global_batch": GB, "frames_per_utterance": Tm}),
        "arith_mode": mode_name, "noise": "on-device Philox4x32-10 (inside the timed region)", "fp16_piece_saturation": bool(saturated),
        "api": "fastdiff_b200.shard.ShardedFastDiff.sample",
        "clocks": clk, "e2e": e2e, "e2e_reference_noise": e2e_ref_noise, "gpu_launches": int(launches), "roofline": roofline, "class_roofline": class_roofline,
        "cpu_baseline": cpu_baseline,
        "load": {"seconds_incl_pack": load_s, "blob_bytes": sh.blob_bytes, "broadcasts": 1 if world > 1 else 0},
        **({"experiment": {"options": args.opt, "nvcc_extra": os.environ.get("FD_NVCC_EXTRA", "")}} if (args.opt or os.environ.get("FD_NVCC_EXTRA")) else {}),
        "kernel_ms_per_step": {k: v["ms"] / args.steps for k, v in per_kernel.items()},
        "ms_per_step_instrumented": ms_instr,
        "kernel_ms_note": "second timed loop of the same K calls with CUDA events around every launch (plain launches in serial order, side stream off, so "
                          "every class is timed alone; `value` comes from the first loop, which replays the library's CUDA graph with the DBlock chain "
                          "overlapping embed / kernel predictor / GEMM on the side stream)",
        "whole_step": whole,
        "limiter": ("per-step: LVC layers of blocks 1/2 (SIMT epilogues + HBM rows), then the kernel_conv GEMM's 2 GB store stream; "
                    "across GPUs: nothing collective in the loop -- the residual is max-over-ranks under sw_power_cap"),
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays, limit):
    """Write each array as float32 `path/<name>.npy`.  An array over `limit` bytes (with --batch / --frames far above the default) is
    replaced by the fixed sample flat[::stride] with the smallest stride that fits, so two builds still compare element for element."""
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        a = t.to(torch.float32).numpy()
        stride = -(-a.nbytes // limit)
        if stride > 1:
            a = a.reshape(-1)[::stride]
        np.save(os.path.join(path, f"{name}.npy"), a)
        log(f"dump: {name} {a.shape} -> {path}" + (f" (flat[::{stride}])" if stride > 1 else ""))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=None, choices=[None, "fp32_simt", "tc_3xtf32", "tc_tf32", "tc_3xf16"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--frames", type=int, default=861)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--opt", action="append", default=[], help="library tuning option key=value (fd_set_option), repeatable")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the waveform the last timed step returned as DIR/audio.npy (float32, at most 64 MB; one file per rank)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
