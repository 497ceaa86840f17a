#!/usr/bin/env python
"""bench.py — benchmark of the per-block audio-graph DSP path (BASELINE.json metric: mono-equivalent samples/s through
the graph at 1/2/4/8 B200; conv-reverb TFLOPS).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--only c2,c3,c4,c5,dag] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic input. ONE JSON line on rank 0:
  headline (`value`, `ms_per_step`, `roofline`, `e2e`, `cpu_baseline`) = c2, BASELINE configs[1]: 1024 stereo voices per GPU,
      gain -> pan -> master-bus sum, 256-frame blocks, 256 blocks per step (weak scaling over ranks, bus exchanged);
  `configs` = the other GPU configs of BASELINE.json, each with its own ms_per_step / value / roofline / e2e / parity:
      c3  4096 voices/GPU, 4-stage biquad cascade + 12000-frame delay line, 512-frame blocks (HBM roofline)
      c4  256 voices/GPU, 48000-tap stereo FIR reverb as a bf16 tcgen05 GEMM (tensor roofline, TFLOP/s)
      c5  65536 sampler voices IN TOTAL (sampler -> gain -> pan -> 4-stage biquad -> FIR reverb -> master bus), sharded
          over the ranks: STRONG scaling of BASELINE configs[4];
      dag a non-chain voice graph (dry + SVF send + biquad send -> 6-port SumNode -> pan -> bus) on the generic lowering, plus block-sized
          calls (one 256-frame block per call) replayed from a captured CUDA graph: us per call;
  `cpu_baseline.c1` = configs[0]: one VolumeNode, mono, 256-frame blocks on the CPU oracle (ns per block of executor plumbing).
Timing: every config runs max(W, 3) untimed warm-up steps, then exactly `--steps` timed steps back to back, bracketed by a
barrier and a stream synchronise on both sides and timed with CUDA events on the processor's stream; the MAX over ranks is
taken. The step count before the last timed step is fixed by the arguments, so stateful configs end in the same state.
`--dump-outputs DIR` writes, per config, the output of the last timed step (what the caller of the timed path receives: the
master bus, or the per-voice outputs) as DIR/<config>.npy (float32, rank 0's); a config whose output exceeds its share of
64 MB keeps a fixed, seeded sample of whole voices (rows of axis 0, in ascending order).
N > 1 is launched by torchrun (one rank per GPU) but uses no torch: the communicator id travels through a file, barriers
and reductions through the product's own NCCL communicator (firewheel_b200/rendezvous.py).
`--impl reference` times the CPU oracle (the C++ restatement of the reference's Rust path — Rust cannot be built in
this image) on all host cores over the headline workload.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import zlib
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))

F32 = np.float32
SR = 48000
C5_TOTAL_VOICES = int(os.environ.get("FW_BENCH_C5_VOICES", "65536"))  # BASELINE configs[4]; the override exists to profile one rank's share (8192) on one GPU
WORKLOADS = {
    # voices per GPU (c5: in total), channels, block frames, blocks per step
    "c1": dict(voices=1, ch=1, block=256, blocks=4096, bus=False, desc="c1: single VolumeNode, mono, 256-frame blocks (CPU plumbing, beep_test shape)"),
    "c2": dict(voices=1024, ch=2, block=256, blocks=256, bus=True, bytes_per_sample=4.004, kernel_class=1, scaling="weak",
               kernel="chain_kernel<VEC=4,CIN=2,BUS,4 voices/warp,16 warps> (gain->pan->bus tree)",
               desc="c2: 1024 stereo voices/GPU, gain->pan->master-bus sum, 256-frame blocks, 256 blocks/step"),
    "c3": dict(voices=4096, ch=2, block=512, blocks=32, bus=False, bytes_per_sample=16.0, kernel_class=3, scaling="weak",
               kernel="biquad_delay_lanes<NS=4,L=4,DELAY,2 rows/lane packed f32x2> (4-stage biquad cascade + 12000-frame delay ring, stage-parallel lanes)",
               desc="c3: 4096 stereo voices/GPU, 4-stage biquad cascade + 12000-frame delay line, 512-frame blocks, 32 blocks/step"),
    "c4": dict(voices=256, ch=2, block=512, blocks=16, bus=False, bytes_per_sample=8.0, kernel_class=3, ir_len=48000, scaling="weak", rotate=16,
               kernel="reverb_gemm_kernel (persistent stream-K, tcgen05.mma kind::f16 M128 N256 K16, 2 TMEM accumulators, TMA 128B-swizzle operands)",
               desc="c4: 256 stereo voices/GPU, FIR convolutional reverb, 48000-tap stereo IR, bf16 tcgen05, 512-frame blocks, 16 blocks/step"),
    "c5": dict(voices=C5_TOTAL_VOICES, ch=2, block=512, blocks=2, bus=True, bytes_per_sample=8.0, kernel_class=3, ir_len=48000, src="sampler", scaling="strong",
               kernel="reverb_gemm_kernel (tcgen05) + biquad_delay_lanes; sampler_kernel source, chain_kernel before and after",
               desc="c5: 65536 looping stereo sampler voices in total (256 two-second f32 resources per GPU, 188 MiB in HBM) -> gain->pan->4-stage biquad->48000-tap FIR reverb->master-bus sum, 512-frame blocks, 2 blocks/step, voices sharded over the ranks"),
}
# a voice graph that is NOT a chain (SURVEY f2): dry + two filtered sends into a 6-port SumNode, then pan and the master bus. It runs on the
# generic per-node lowering (one launch group per scheduled node over the reference's own buffer assignment) and, for block-sized calls, on CUDA-graph replay.
WORKLOADS["dag"] = dict(voices=1024, ch=2, block=256, blocks=64, bus=True, bytes_per_sample=4.004, kernel_class=-1, scaling="weak",
                        kernel="generic lowering: chain_kernel (gain / pan / copies), biquad_delay_lanes (SVF, biquad), sum_kernel, bus tree",
                        desc="dag: 1024 stereo voices/GPU, graph_in -> {gain | 2-stage SVF -> gain | 2-stage biquad -> gain} -> 6-port SumNode -> pan -> master bus, 256-frame blocks, 64 blocks/step")
REVERB_WORKLOADS = ("c4", "c5")
DUMP_LIMIT_BYTES = 64_000_000  # all --dump-outputs files of one run together


def synth(shape, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    r = rng.integers(0, 1 << 24, size=shape, dtype=np.uint32)
    return (r.astype(F32) * F32(2.0 ** -23) - F32(1.0)).astype(F32)


def voice_params(V, seed):
    rng = np.random.default_rng(seed)
    return (25 + 75 * rng.random(V)).astype(F32), rng.uniform(-1, 1, V).astype(F32)  # SURVEY §8d: never muted


def biquad_params(fw, lib, V, seed):
    """SURVEY §8d: RBJ low-pass / peaking, fc log-uniform 200 Hz - 8 kHz, Q in [0.5, 2] at 48 kHz."""
    rng = np.random.default_rng(seed)
    k = np.zeros((V, 4, 5), F32)
    for v in range(V):
        for s in range(4):
            k[v, s] = fw.design_rbj(lib, 0 if s % 2 == 0 else 4, 200.0 * 40.0 ** rng.random(), rng.uniform(0.5, 2.0), rng.uniform(-3, 3), SR)
    return k


def reverb_ir(L):
    rng = np.random.default_rng(0x1200)
    ir = rng.standard_normal((2, L)) * np.exp(-6.9 * np.arange(L) / L)  # SURVEY §8d
    return (ir / np.sqrt((ir ** 2).sum(axis=1, keepdims=True))).astype(F32)


def build_graph(fw, lib, workload, V, block, device, seed):
    """The voice graph of a workload, on `lib` (the CUDA product, or the CPU oracle for the baseline / parity legs)."""
    w = WORKLOADS[workload]
    sampler_src = w.get("src") == "sampler"
    cx = fw.FirewheelGraphCtx(lib, fw.AudioGraphConfig(num_graph_inputs=0 if sampler_src else w["ch"], num_graph_outputs=w["ch"], num_voices=V,
                                                       master_bus=w["bus"], device=device, max_call_frames=w["block"] * w["blocks"]))  # one step = one chunk
    g = cx.graph
    C = w["ch"]
    if workload == "c1":
        nodes = [g.add_node(1, 1, fw.VolumeNode(70.0))]
    elif workload == "c2":
        pct, pan = voice_params(V, seed)
        nodes = [g.add_node(2, 2, fw.VolumeNode(100.0)), g.add_node(2, 2, fw.PanNode(0.0))]
        g.set_percent_volume(nodes[0], pct)
        g.set_pan(nodes[1], pan)
    elif workload == "dag":
        pct, pan = voice_params(V, seed)
        gin, gout = g.graph_in_node(), g.graph_out_node()
        dry, svf, wet1, bq, wet2 = (g.add_node(2, 2, fw.VolumeNode(80.0)), g.add_node(2, 2, fw.SvfNode(2)), g.add_node(2, 2, fw.VolumeNode(40.0)),
                                    g.add_node(2, 2, fw.BiquadNode(2)), g.add_node(2, 2, fw.VolumeNode(30.0)))
        mix, pn = g.add_node(6, 2, fw.SumNode()), g.add_node(2, 2, fw.PanNode(0.0))
        g.set_percent_volume(dry, pct); g.set_pan(pn, pan)
        g.set_svf_coeffs(svf, np.stack([[fw.design_svf(lib, 0, 1200.0, 0.8, SR), fw.design_svf(lib, 4, 3000.0, 1.2, SR)] for _ in range(V)]).astype(F32))
        g.set_biquad_coeffs(bq, biquad_params(fw, lib, V, seed)[:, :2].copy())
        for c in range(2):
            g.connect(gin, c, dry, c, False); g.connect(gin, c, svf, c, False); g.connect(gin, c, bq, c, False)
            g.connect(svf, c, wet1, c, False); g.connect(bq, c, wet2, c, False)
            g.connect(dry, c, mix, c, False); g.connect(wet1, c, mix, 2 + c, False); g.connect(wet2, c, mix, 4 + c, False)
            g.connect(mix, c, pn, c, False); g.connect(pn, c, gout, c, False)
        proc = cx.activate(SR, C, C, block)
        if proc is None:
            raise RuntimeError("activate failed")
        st = cx.update()
        if st.graph_error is not None:
            raise RuntimeError(f"compile failed: {st.graph_error} {cx.last_error()}")
        return cx, proc
    elif workload in REVERB_WORKLOADS:
        nodes = [g.add_node(2, 2, fw.ConvReverbNode(reverb_ir(w["ir_len"])))]
        if workload == "c5":
            pct, pan = voice_params(V, seed)
            pre = [g.add_node(2, 2, fw.VolumeNode(100.0)), g.add_node(2, 2, fw.PanNode(0.0)), g.add_node(2, 2, fw.BiquadNode(4))]
            g.set_percent_volume(pre[0], pct); g.set_pan(pre[1], pan); g.set_biquad_coeffs(pre[2], biquad_params(fw, lib, V, seed))
            nodes = pre + nodes
    else:
        nodes = [g.add_node(2, 2, fw.BiquadNode(4)), g.add_node(2, 2, fw.DelayNode(12000))]
        g.set_biquad_coeffs(nodes[0], biquad_params(fw, lib, V, seed))
    smp = None
    if sampler_src:
        smp = g.add_node(0, 2, fw.SamplerNode(100.0))
        prev = smp
    else:
        prev = g.graph_in_node()
    for n in nodes + [g.graph_out_node()]:
        for c in range(C):
            g.connect(prev, c, n, c, False)
        prev = n
    proc = cx.activate(SR, 0 if sampler_src else C, C, block)
    if proc is None:
        raise RuntimeError("activate failed")
    st = cx.update()
    if st.graph_error is not None:
        raise RuntimeError(f"compile failed: {st.graph_error} {cx.last_error()}")
    if sampler_src:
        # 256 two-second stereo f32 resources (188 MiB: larger than L2); voice v loops resource v % n_res from its own offset
        n_res = min(256, V)
        handles = [g.create_sample_resource(synth((2, 2 * SR), 0x5A000000 + (seed % 4096) * 4096 + r)) for r in range(n_res)]
        for v in range(V):
            g.sampler_set_sample(smp, handles[v % n_res], True, voice=v)
            g.sampler_set_loop_range(smp, "full", voice=v)
            g.sampler_set_playhead(smp, ((v // n_res) * 2731 % (2 * SR)) / SR, voice=v)
        g.sampler_play(smp)
    return cx, proc


# ---- clocks (B200_PROFILING.md: sample DURING the timed region) ---------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.rows, self.stop_evt, self.th = gpu_index, [], threading.Event(), None

    def _once(self):
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                 capture_output=True, text=True, timeout=5).stdout.strip()
            if out:
                self.rows.append([c.strip() for c in out.split(",")])
                return
        except Exception:
            pass
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            f = lambda bit: "Active" if r & bit else "Not Active"
            self.rows.append([str(self.idx), str(sm), str(mx), "0", f(0x8), f(0x40), f(0x20), f(0x4)])
        except Exception:
            pass

    def start(self):
        def loop():
            while not self.stop_evt.is_set():
                self._once()
                self.stop_evt.wait(0.1)
        self.th = threading.Thread(target=loop, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_evt.set()
        if self.th:
            self.th.join(timeout=10)
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6), ("sw_power_cap", 7)):
                if len(r) > col and r[col] == "Active":
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm": (float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"),
                "tensor": (float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst)"),
                "tensor_sustained": float(d.get("bf16_tflops_sustained", 0.0)) or None}
    return {"hbm": (6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"), "tensor": (1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s)"), "tensor_sustained": None}


def cfg_dict(workload, V, world):
    """The `config` object: identical for the product arm and the reference arm of the same workload."""
    w = WORKLOADS[workload]
    T, C = w["block"] * w["blocks"], w["ch"]
    in_mib = (V * (0 if w.get("src") == "sampler" else C) * T * 4) >> 20
    if w.get("src") == "sampler":
        l2 = "sample pool larger than L2 (188 MiB per GPU), every voice at its own offset"
    elif w.get("rotate"):
        l2 = f"inputs rotate over {w['rotate']} buffers of {in_mib} MiB ({w['rotate'] * in_mib} MiB, larger than L2)"
    else:
        l2 = f"inputs larger than L2 ({in_mib} MiB per GPU per step)"
    return {"workload": w["desc"], "voices_per_gpu": V, "channels": C, "block_frames": w["block"], "blocks_per_step": w["blocks"],
            "l2": l2, "layout": "planar [voice][ch][frame]", "parallelism": f"voices sharded over {world} rank(s)"}


# ---- CPU oracle legs ---------------------------------------------------------------------------------
def oracle_rate(V, block, n_blocks, threads, seed=7, steps=1, warmup=0, workload="c2"):
    """Mono-equivalent samples/s of the CPU oracle on V voices x n_blocks blocks, voices split over `threads`
    replicas (each a disjoint voice range with its own partial bus; the reference itself is single-threaded)."""
    import firewheel_b200 as fw
    import pyoracle
    lib = pyoracle.load()
    w = WORKLOADS[workload]
    T, C = block * n_blocks, w["ch"]
    bus = w["bus"]
    bounds = np.linspace(0, V, threads + 1).astype(int)
    parts = []
    for i in range(threads):
        lo, hi = bounds[i], bounds[i + 1]
        if hi <= lo:
            continue
        cx, proc = build_graph(fw, lib, workload, hi - lo, block, 0, seed * 100 + i)
        x = synth((hi - lo, 0 if w.get("src") == "sampler" else C, T), seed * 1000 + i)
        out = np.zeros((C, T) if bus else (hi - lo, C, T), F32)
        parts.append((cx, proc, x, out))

    def run(p):
        cx, proc, x, out = p
        rc, _ = proc.process_planar(x, out, x.shape[1], C, T)
        assert rc == 0

    pool = ThreadPoolExecutor(len(parts)) if len(parts) > 1 else None  # persistent: thread start-up is not the reference's cost

    def one_step():
        if pool is None:
            run(parts[0])
        else:
            list(pool.map(run, parts))
            if bus:
                mix = parts[0][3].copy()
                for p in parts[1:]:
                    mix += p[3]  # top of the mix tree over replicas
    for _ in range(warmup):
        one_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = time.perf_counter() - t0
    if pool is not None:
        pool.shutdown()
    for cx, proc, _, _ in parts:
        proc.free(); cx.update(); cx.free()
    return V * C * T * steps / dt, dt / steps


def run_reference(args, rank, world):
    if rank != 0:
        return
    w = WORKLOADS["c2"]
    cores = os.cpu_count() or 1
    V = w["voices"] * max(args.gpus, 1)
    n_blocks = w["blocks"]  # the full step (a few ms per replica thread), so dispatch overhead does not flatter the GPU
    val, sec_per_step = oracle_rate(V, w["block"], n_blocks, cores, steps=args.steps, warmup=args.warmup, workload="c2")
    sample = f"{V} voices x {n_blocks} of {w['blocks']} blocks per step, {cores} replica threads over disjoint voice ranges"
    line = {"impl": "reference", "metric": "mono_equiv_samples_per_sec", "value": val, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg_dict("c2", w["voices"], max(args.gpus, 1)),
            "note": "CPU oracle = C++ restatement of the reference's Rust path (no Rust toolchain in this image); the reference itself is single-threaded, the replicas are a courtesy",
            "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_leg(workload, V, F, KB):
    """Single-thread CPU oracle on a bounded sample of the workload (~10 s of CPU work); the reference's execution model."""
    n_blocks = 64 if workload == "c2" else 2
    Vc = V if workload not in REVERB_WORKLOADS else 2  # the direct-form FIR oracle needs ~0.2 s per voice-block
    if workload in REVERB_WORKLOADS:
        n_blocks = 1
    if workload == "c5":
        Vc = 2
    rate, sec = oracle_rate(Vc, F, n_blocks, 1, steps=1, warmup=0, workload=workload)
    if sec < 2.0 and workload not in REVERB_WORKLOADS:  # size the sample towards ~10 s of CPU work
        n_blocks = int(min(KB * 8, max(n_blocks, n_blocks * 10.0 / max(sec, 1e-3))))
        rate, sec = oracle_rate(Vc, F, n_blocks, 1, steps=1, warmup=0, workload=workload)
    elif workload in REVERB_WORKLOADS and sec < 5.0:
        Vc = int(min(64, max(2, Vc * 10.0 / max(sec, 1e-3))))
        rate, sec = oracle_rate(Vc, F, n_blocks, 1, steps=1, warmup=0, workload=workload)
    return {"value": rate, "unit": "samples/s", "cores": 1, "kind": "port",
            "sample": f"{Vc} voices x {n_blocks} blocks of {F} frames, 1 thread (the reference's execution model), {sec:.1f} s"}


def c1_leg():
    """BASELINE configs[0]: one VolumeNode between a mono source and graph_out, F = 256, CPU oracle: ns per block of executor plumbing."""
    import firewheel_b200 as fw
    import pyoracle
    lib = pyoracle.load()
    w = WORKLOADS["c1"]
    cx, proc = build_graph(fw, lib, "c1", 1, w["block"], 0, 1)
    T = w["block"] * w["blocks"]
    x = synth((1, 1, T), 5)
    out = np.zeros((1, 1, T), F32)
    proc.process_planar(x, out, 1, 1, T)
    reps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < 1.0:
        rc, _ = proc.process_planar(x, out, 1, 1, T)
        assert rc == 0
        reps += 1
    dt = time.perf_counter() - t0
    proc.free(); cx.update(); cx.free()
    blocks = reps * w["blocks"]
    return {"ns_per_block": dt / blocks * 1e9, "value": blocks * w["block"] / dt, "unit": "samples/s", "cores": 1, "kind": "port",
            "sample": f"{blocks} blocks of 256 mono frames through graph_in -> VolumeNode -> graph_out, {dt:.1f} s"}


def tree_sum(parts):
    """Balanced binary tree over per-rank buses, neighbours (2i, 2i+1) per level, an unpaired last element carried up."""
    parts = [p.copy() for p in parts]
    while len(parts) > 1:
        nxt = []
        for i in range(0, len(parts) - 1, 2):
            nxt.append((parts[i] + parts[i + 1]).astype(F32))
        if len(parts) % 2:
            nxt.append(parts[-1])
        parts = nxt
    return parts[0]


# ---- the product arm ---------------------------------------------------------------------------------
class Comm:
    """Barrier / reductions over the current processor's communicator (NCCL); trivial for one rank."""

    def __init__(self, proc, rank, world):
        self.proc, self.rank, self.world = proc, rank, world

    def gather(self, a):
        a = np.ascontiguousarray(a)
        return self.proc.comm_allgather(a) if self.world > 1 else a[None]

    def barrier(self):
        self.proc.sync()
        if self.world > 1:
            self.gather(np.zeros(1, np.int64))

    def max(self, a):
        return self.gather(np.asarray(a, np.float64)).max(axis=0)


def dump_output(out_dir, name, y, limit):
    """`y` as out_dir/<name>.npy; above `limit` bytes, a seeded sample of its rows (voices) in ascending order."""
    out_dir.mkdir(parents=True, exist_ok=True)
    if y.nbytes > limit:
        n = max(1, limit // (y.nbytes // y.shape[0]))
        y = y[np.sort(np.random.default_rng(0).choice(y.shape[0], n, replace=False))]
    np.save(out_dir / f"{name}.npy", np.ascontiguousarray(y, F32))


def run_config(fw, lib, name, args, rank, world, local_rank, want_cpu, dump_bytes):
    from firewheel_b200 import rendezvous
    w = WORKLOADS[name]
    C, F, KB = w["ch"], w["block"], w["blocks"]
    V = w["voices"] // world if w["scaling"] == "strong" else w["voices"]
    T = F * KB
    cx, proc = build_graph(fw, lib, name, V, F, local_rank, 1000 + rank)
    rendezvous.init_comm(lib, proc, rank, world)  # every config gets the communicator: the bus exchange (c2, c5) and the harness's barriers use it
    comm = Comm(proc, rank, world)
    Cin = 0 if w.get("src") == "sampler" else C  # sampler voices read their sample resources from HBM, not a stream input
    in_bytes = V * Cin * T * 4
    out_bytes = C * T * 4 if w["bus"] else V * C * T * 4
    n_rot = w.get("rotate", 1) if in_bytes else 1

    h_in = lib.host_alloc_pinned(in_bytes) if in_bytes else 0
    h_out = lib.host_alloc_pinned(out_bytes)
    if (in_bytes and not h_in) or not h_out:
        raise RuntimeError("pinned allocation failed")
    if in_bytes:
        x = np.ctypeslib.as_array(ctypes.cast(h_in, ctypes.POINTER(ctypes.c_float)), shape=(V, C, T))
    y = np.ctypeslib.as_array(ctypes.cast(h_out, ctypes.POINTER(ctypes.c_float)), shape=(C, T) if w["bus"] else (V, C, T))
    d_ins = [lib.dev_malloc(local_rank, in_bytes) if in_bytes else 0 for _ in range(n_rot)]
    d_out = lib.dev_malloc(local_rank, out_bytes)
    if (in_bytes and not all(d_ins)) or not d_out:
        raise RuntimeError("device allocation failed: " + lib.last_device_error().decode())
    for r in (range(n_rot - 1, -1, -1) if in_bytes else ()):  # the last upload (rotation slot 0) stays in the pinned buffer for the e2e / parity legs
        chunk = 64
        for v0 in range(0, V, chunk):
            x[v0:v0 + chunk] = synth((min(chunk, V - v0), C, T), 0xF17E0000 + rank * 65536 + r * 4096 + v0)
        proc.h2d(d_ins[r], h_in, in_bytes)
        proc.sync()

    # ---- parity of the timed configuration, on the context's fresh state: a 4-block prefix against the CPU oracle ----
    parity = parity_prefix(fw, lib, name, proc, comm, x if in_bytes else None, d_ins[0], d_out, h_out, y, V, C, F, rank, world)

    step_i = [0]

    def step():
        rc = proc.process_planar_device(d_ins[step_i[0] % n_rot], d_out, Cin, C, T)
        step_i[0] += 1
        if rc != 0:
            raise RuntimeError(f"{name}: process_planar_device rc={rc} {lib.last_device_error().decode()}")

    def one_pass(k):
        comm.barrier()
        proc.event_record(0)
        for _ in range(k):
            step()
        proc.event_record(1)
        proc.sync()
        return proc.event_elapsed_ms(0, 1)

    for _ in range(max(args.warmup, 3)):
        step()
    clocks = ClockSampler(local_rank)
    clocks.start()
    launches0 = proc.kernel_launches()
    mine = one_pass(args.steps)
    launches = proc.kernel_launches() - launches0
    clk = clocks.stop()
    if dump_bytes and rank == 0:
        proc.d2h(h_out, d_out, out_bytes)
        proc.sync()
        dump_output(Path(args.dump_outputs), name, y, dump_bytes)
    timed_ms = float(comm.max([mine])[0])
    by_rank = [float(v) / args.steps for v in comm.gather(np.array([mine], np.float64))[:, 0]]  # GPUs of one box differ
    ms_per_step = timed_ms / args.steps
    samples_per_step = V * C * T * world
    value = samples_per_step / (ms_per_step * 1e-3)

    # per-kernel-class pass: a CUDA-event pair around every kernel class (these events serialise the programmatic-dependent-
    # launch overlap, so they stay out of the timed window)
    proc.profile(True)
    prof_steps = max(args.steps, 5)
    for _ in range(prof_steps):
        step()
    prof_ms, prof_n = proc.profile_read()
    proc.profile(False)

    proc.d2h(h_out, d_out, out_bytes)
    proc.sync()
    if not (np.all(np.isfinite(y[..., ::97])) and float(np.abs(y[..., ::97]).max()) > 0.0):
        raise RuntimeError(f"{name}: output is not finite / all zero")
    ranks_identical = None
    if world > 1 and w["bus"]:  # the master bus must be the same bits on every rank
        crc = np.array([zlib.crc32(y.tobytes())], np.int64)
        allc = comm.gather(crc)
        ranks_identical = bool((allc == allc[0]).all())

    # ---- end-to-end: host buffers through the C-ABI call, H2D + D2H inside the timed region ----
    e2e_steps = min(args.steps, 10)
    for _ in range(2):
        rc, _ = proc.process_planar(h_in, h_out, Cin, C, T)
        assert rc == 0
    comm.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        rc, _ = proc.process_planar(h_in, h_out, Cin, C, T)
        assert rc == 0
    proc.sync()
    e2e_s = float(comm.max([(time.perf_counter() - t0) / e2e_steps])[0])

    # ---- roofline of the dominant kernel class, CUDA events on the launching stream ----
    pk = peaks()
    kc = w["kernel_class"]
    kernel_ms = (sum(prof_ms) if kc < 0 else prof_ms[kc]) / prof_steps  # all launches of the dominant kernel class in one step (dag: of every class)
    kernel_ms = min(kernel_ms, ms_per_step)  # the event pairs of the profiling pass add launch gaps: a class cannot take longer than the step it is part of
    tensor = name in REVERB_WORKLOADS
    # SURVEY §8d: c2 reads V*C*T f32 and writes the C*T bus; c3 moves in + out + delay-ring read + write = 16 B/sample
    algo_bytes = 4 * C * T * (V + 1) if name in ("c2", "dag") else int(w["bytes_per_sample"] * V * C * T)
    flops = 2.0 * w["ir_len"] * V * C * T if tensor else None
    if tensor:
        peak, peak_src = pk["tensor"]
        achieved = flops / (kernel_ms * 1e-3) / 1e12 if kernel_ms > 0 else 0.0
    else:
        peak, peak_src = pk["hbm"]
        achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
    traffic = None
    tp = ROOT / "profiles" / f"r02_{name}_traffic.json"
    if not tp.exists():
        tp = ROOT / "profiles" / f"r02_{name}_tensor.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "tensor" if tensor else "hbm", "kernel": w["kernel"], "achieved": achieved, "peak": peak, "unit": "TFLOP/s" if tensor else "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "kernel_ms": kernel_ms,
                "kernel_ms_note": "second pass with a CUDA-event pair around every kernel class (PDL overlap off); sum over the class's launches in one step, capped at the timed step",
                "algorithmic_bytes_per_launch": None if tensor else algo_bytes, "algorithmic_flops_per_launch": flops,
                "step_level_frac": ((flops / (ms_per_step * 1e-3) / 1e12) if tensor else (algo_bytes / (ms_per_step * 1e-3) / 1e9)) / peak,
                "step_share": {"control_ms": prof_ms[0] / prof_steps, "chain_ms": prof_ms[1] / prof_steps,
                               "combine_ms": prof_ms[2] / prof_steps, "temporal_ms": prof_ms[3] / prof_steps}}
    if tensor:
        roofline["tflops_step_level"] = flops / (ms_per_step * 1e-3) / 1e12  # per GPU, whole step (prepare + GEMM + neighbours)
        roofline["frac_of_sustained_peak"] = (achieved / pk["tensor_sustained"]) if pk["tensor_sustained"] else None

    cpu = cpu_leg(name, V, F, KB) if (want_cpu and rank == 0) else None
    block_call = None
    if name == "dag":  # the interactive shape: one block per call, the same buffers every time -> captured once, then one cudaGraphLaunch per call
        n_calls = 2000
        for _ in range(8):
            proc.process_planar_device(d_ins[0], d_out, Cin, C, F)
        proc.sync()
        r0, l0 = proc.graph_replays(), proc.kernel_launches()
        t0 = time.perf_counter()
        proc.event_record(0)
        for _ in range(n_calls):
            proc.process_planar_device(d_ins[0], d_out, Cin, C, F)
        proc.event_record(1)
        proc.sync()
        wall = time.perf_counter() - t0
        block_call = {"frames_per_call": F, "calls": n_calls, "us_per_call_device": proc.event_elapsed_ms(0, 1) * 1e3 / n_calls, "us_per_call_host": wall * 1e6 / n_calls,
                      "graph_replays": proc.graph_replays() - r0, "kernels_per_call": (proc.kernel_launches() - l0) / n_calls,
                      "note": "256-frame block for 1024 voices per call through fw_processor_process_planar_device; realtime budget of one block at 48 kHz is 5333 us"}

    res = {"metric": "mono_equiv_samples_per_sec", "value": value, "unit": "samples/s", "ms_per_step": ms_per_step,
           "ms_per_step_by_rank": by_rank, "timed_steps": args.steps, "timed_seconds": timed_ms * 1e-3,
           "scaling": w["scaling"], "dtype": "bf16 x bf16 -> f32 (FIR), f32 elsewhere" if tensor else "f32",
           "config": cfg_dict(name, V, world), "clocks": clk,
           "e2e": {"value": samples_per_step / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": in_bytes * world, "d2h_bytes_per_step": out_bytes * world,
                   "steps": e2e_steps, "ms_per_step": e2e_s * 1e3, "api": "fw_processor_process_planar (pinned host buffers)"},
           "gpu_launches_timed": int(launches), "roofline": roofline, "parity": parity, "cpu_baseline": cpu}
    if block_call:
        res["block_sized_calls"] = block_call
    if tensor:
        res["tflops"] = flops * world / (ms_per_step * 1e-3) / 1e12
    if world > 1 and w["bus"]:
        res["exchange"] = "NCCL all-gather on a high-priority side stream (device-word hand-over, no event on the main stream) + rank-ordered tree"
        res["bus_identical_on_all_ranks"] = ranks_identical
        if parity and "bus" in parity:
            res["bus_parity"] = parity["bus"] if ranks_identical else "mismatch"
    comm.barrier()
    proc.free()
    cx.update()
    cx.free()
    for d in d_ins:
        if d:
            lib.dev_free(local_rank, d)
    lib.dev_free(local_rank, d_out)
    if h_in:
        lib.host_free_pinned(h_in)
    lib.host_free_pinned(h_out)
    return res


def parity_prefix(fw, lib, name, proc, comm, x, d_in, d_out, h_out, y, V, C, F, rank, world):
    """First call on the fresh context: 4 blocks, compared with the CPU oracle before anything else advances the state.
    c2: bit-exact, and across ranks against the oracle's tree of per-rank buses. c3: bit-exact per voice. c4: voices 0-1 within 1e-5
    of the bf16-rounded oracle (the direct-form FIR costs 96 kflop per sample on the CPU). c5: the bus mixes every voice, the
    oracle cannot render it in bench time: cross-rank identity only (tests/ hold its small-size parity)."""
    import pyoracle
    if name == "c5":
        return {"checked": "cross-rank identity of the master bus only (small-size parity: tests/test_gpu_parity.py, test_gpu_sampler.py)"}
    olib = pyoracle.load()
    w = WORKLOADS[name]
    Tp = 4 * F
    T = F * w["blocks"]
    xp = np.ascontiguousarray(x[:, :, :Tp])
    # product: 4 blocks read in place from the resident step input (row pitch T != frames is not an API notion: use a compact copy)
    d_pre = lib.dev_malloc(proc_device(proc), xp.nbytes)
    h_pre = lib.host_alloc_pinned(xp.nbytes)
    np.ctypeslib.as_array(ctypes.cast(h_pre, ctypes.POINTER(ctypes.c_float)), shape=xp.shape)[...] = xp
    proc.h2d(d_pre, h_pre, xp.nbytes)
    out_elems = (C * Tp) if w["bus"] else (V * C * Tp)
    d_o = lib.dev_malloc(proc_device(proc), out_elems * 4)
    rc = proc.process_planar_device(d_pre, d_o, C, C, Tp)
    got = np.zeros((C, Tp) if w["bus"] else (V, C, Tp), F32)
    h_o = lib.host_alloc_pinned(got.nbytes)
    proc.d2h(h_o, d_o, got.nbytes)
    proc.sync()
    got[...] = np.ctypeslib.as_array(ctypes.cast(h_o, ctypes.POINTER(ctypes.c_float)), shape=got.shape)
    for p in (h_pre, h_o):
        lib.host_free_pinned(p)
    for d in (d_pre, d_o):
        lib.dev_free(proc_device(proc), d)
    if rc != 0:
        return {"error": f"prefix call rc={rc}"}
    Vo = V if name != "c4" else 2
    ocx, oproc = build_graph(fw, olib, name, Vo, F, 0, 1000 + rank)
    ref = np.zeros((C, Tp) if w["bus"] else (Vo, C, Tp), F32)
    orc, _ = oproc.process_planar(np.ascontiguousarray(xp[:Vo]), ref, C, C, Tp)
    oproc.free(); ocx.update(); ocx.free()
    if name == "c4":
        err = float(np.abs(got[:Vo].astype(np.float64) - ref.astype(np.float64)).max() / max(float(np.abs(ref).max()), 1e-30))
        return {"voices_checked": Vo, "frames": Tp, "max_err_over_max_abs": err, "tolerance": 1e-5, "ok": bool(err <= 1e-5)}
    if w["bus"]:
        parts = comm.gather(ref)
        want = tree_sum(list(parts))
        ok = bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)))
        return {"frames": Tp, "bus": "bit-exact" if ok else "mismatch", "ok": ok,
                "against": f"tree_sum of the {world} per-rank CPU-oracle buses (each {V} voices)"}
    ok = bool(np.array_equal(got.view(np.uint32), ref.view(np.uint32)))
    return {"frames": Tp, "voices_checked": V, "bits": "bit-exact" if ok else "mismatch", "ok": ok}


def proc_device(proc):
    return int(os.environ.get("LOCAL_RANK", "0"))


def run_b200(args, rank, world, local_rank):
    import firewheel_b200 as fw
    from firewheel_b200 import rendezvous
    lib = fw.load()  # raises if the CUDA library is missing: no CPU fallback
    if lib.device_count() <= local_rank:
        raise RuntimeError("no CUDA device for this rank: " + lib.last_device_error().decode())
    if world > 1:
        # NCCL prints its version banner on stdout at NCCL_DEBUG >= VERSION; keep stdout for the single JSON line
        os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ["NCCL_DEBUG"] = "NONE"
    names = [n for n in args.only.split(",") if n]
    want_cpu = world == 1 and not os.environ.get("FW_BENCH_SKIP_CPU")
    dump_bytes = DUMP_LIMIT_BYTES // len(names) - 4096 if args.dump_outputs else 0  # 4096: room for the .npy header
    results = {}
    for n in names:
        t0 = time.perf_counter()
        results[n] = run_config(fw, lib, n, args, rank, world, local_rank, want_cpu, dump_bytes)
        results[n]["bench_wall_s"] = time.perf_counter() - t0
    rendezvous.cleanup(rank)
    if rank != 0:
        return
    head_name = "c2" if "c2" in results else names[0]
    head = results.pop(head_name)
    line = {"metric": "mono_equiv_samples_per_sec", "value": head["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": head["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": head["config"], "clocks": head["clocks"], "e2e": head["e2e"],
            "gpu_launches": head["gpu_launches_timed"], "roofline": head["roofline"], "cpu_baseline": head["cpu_baseline"]}
    for k in ("ms_per_step_by_rank", "timed_seconds", "parity", "exchange", "bus_parity", "bus_identical_on_all_ranks", "block_sized_calls"):
        if k in head:
            line[k] = head[k]
    if want_cpu and line["cpu_baseline"] is not None:
        line["cpu_baseline"]["c1"] = c1_leg()
    line["configs"] = results
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--only", default="c2,c3,c4,c5,dag", help="comma-separated configs to run (the first of c2 / the list is the headline)")
    ap.add_argument("--workload", default=None, help="alias of --only for a single config")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", dest="dump_outputs",
                    help="write each config's output of the last timed step to DIR/<config>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.workload:
        args.only = args.workload
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
