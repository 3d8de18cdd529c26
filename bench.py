#!/usr/bin/env python
"""Benchmark of the whisper-burn hot path on B200 (contract: see the task statement / DESIGN.md section 6).

    python bench.py --gpus 1 --steps 5 --warmup 3                 # our arm  (C ABI -> sm_100a kernels)
    python bench.py --impl reference --gpus 1 --steps 1 --warmup 0  # reference arm: CPU oracle, reference-cost mode
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): audio-seconds/sec.  A "step" = one pass of the hot path (log-mel -> encoder ->
cross K/V -> greedy decode to EOT or 100 steps) over this rank's batch of synthetic 30 s chunks.

ONE JSON line.  Its top-level fields are the HEADLINE workload = BASELINE configs[1]: tiny.en, ONE 30 s chunk
(3 reference windows, SURVEY F6), greedy; `configs` carries, measured in the same run with the same method, every
workload of --configs (default: the headline, then BASELINE configs[2] = small.en with 8 chunks batched, fp32 and
fp16 K/V cache), each with its own value / e2e / roofline.
N>1: weak scaling, every rank decodes its own chunk(s) (no data-path collective), then ONE NCCL all-gather of the
token buffers (device tensors, one pinned D2H); value = 30 s * total chunks / max-over-ranks step time.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CHUNK_SAMPLES = 480000
CHUNK_SECONDS = 30.0
DEFAULT_CONFIGS = "tiny.en:1:f32,small.en:8:f32,small.en:8:f16,tiny.en:1:f16"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--configs", default=None, help="comma list of model:chunks_per_gpu:kv; the first one is the headline "
                                                    f"(default {DEFAULT_CONFIGS})")
    ap.add_argument("--model", default=None, help="shorthand for --configs MODEL:CHUNKS:KV")
    ap.add_argument("--chunks-per-gpu", type=int, default=1)
    ap.add_argument("--kv", default="f32", choices=["f32", "f16"], help="K/V cache dtype (f32 = reference numerics)")
    ap.add_argument("--beam", type=int, default=1)
    ap.add_argument("--max-depth", type=int, default=100)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-windows", type=int, default=0, help="windows of chunk 0 timed on the CPU (0 = all)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the token ids of the last timed step of every workload to DIR/<name>.npy (float64)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.configs is None:
        a.configs = f"{a.model}:{a.chunks_per_gpu}:{a.kv}" if a.model else DEFAULT_CONFIGS
    a.config_list = []
    for item in a.configs.split(","):
        parts = item.split(":")
        a.config_list.append((parts[0], int(parts[1]) if len(parts) > 1 else 1, parts[2] if len(parts) > 2 else "f32"))
    return a


def host_cores() -> int:
    """Threads the CPU arm can really use: affinity mask capped by the cgroup CPU quota (the GPU
    boxes expose 128 logical CPUs under a 16-CPU quota; oversubscribing MKL there is ~100x slower)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    return max(1, n)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def workload_name(model: str, chunks: int, beam: int, depth: int) -> str:
    """The same string in both arms (the driver compares it)."""
    return (f"{model}, {chunks}x30 s synthetic 16 kHz chunk(s) per GPU, R-mode (3 reference windows per chunk), "
            f"greedy (beam {beam}), max_depth {depth}")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_pass(beam, depth, dims, w_t, sp, chunk, n_windows: int):
    """The reference's own CPU path restated (oracle, reference-cost mode: no KV cache, full-prefix
    recompute, all-position logits, per-window DFT/filterbank rebuild) on windows of one chunk."""
    import torch
    from oracle import audio as o_audio, transcribe as o_tr  # CPU-baseline leg only
    window_len = o_audio.max_waveform_samples(dims.n_audio_ctx - o_tr.PADDING)
    bounds = o_tr.window_bounds(len(chunk), 16000, window_len)
    if n_windows > 0:
        bounds = bounds[:n_windows]
    t0 = time.perf_counter()
    n_tok = 0
    for (s, e) in bounds:
        mel = o_audio.prep_audio(torch.from_numpy(np.ascontiguousarray(chunk[s:e]))[None])
        toks = o_tr.mels_to_tokens(w_t, dims, sp, mel, beam_size=beam, max_depth=depth, use_cache=False)
        n_tok += len(toks)
    dt = time.perf_counter() - t0
    # audio covered by the sample: windows overlap by 3 s; count the span they cover
    span = (bounds[-1][1] - bounds[0][0]) / 16000.0
    return span, dt, len(bounds), n_tok


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the Rust/libtorch
    original cannot be built here: no cargo/rustc, un-vendored crates) on this box's host cores, on the
    HEADLINE workload of our arm (first entry of --configs)."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import synth
    model, chunks, _ = args.config_list[0]
    torch.set_num_threads(host_cores())
    dims, w_np, w_t = synth.make_weights(model, seed=0)
    sp = synth.special_tokens(dims)
    chunk = synth.chunk_waveform(0, CHUNK_SAMPLES)
    nwin = args.cpu_baseline_windows
    for _ in range(args.warmup):
        cpu_reference_pass(args.beam, args.max_depth, dims, w_t, sp, chunk, 1)
    times, span = [], None
    for _ in range(args.steps):
        span, dt, nw, _ = cpu_reference_pass(args.beam, args.max_depth, dims, w_t, sp, chunk, nwin)
        times.append(dt)
    ms = 1000.0 * float(np.mean(times))
    val = span / (ms / 1000.0)
    sample = f"{nw} of 3 reference windows of chunk 0 ({span:.2f} s of audio), greedy depth {args.max_depth}, no KV cache"
    line = {
        "impl": "reference", "metric": "audio-seconds/sec", "value": val, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(model, chunks, args.beam, args.max_depth),
                   "path": "CPU reference-cost path (oracle port of the reference's libtorch-CPU fp32 semantics, no KV cache)",
                   "sample": sample},
        "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def algorithmic_bytes(dims, window_lens, wbytes: int, kvb: int, steps: int) -> int:
    """SURVEY.md 8d bytes of ONE persistent-decoder launch (3 prompt positions without logits + `steps` greedy positions) over the
    windows of `window_lens` samples: decoder weights once per position for the whole batch, the vocabulary matrix on the positions
    that produce logits, every window's cross K/V per position, every row's self K/V up to the current position."""
    d, V, L, R = dims.n_text_state, dims.n_vocab, dims.n_text_layer, len(window_lens)
    n_pos = steps + 3
    T_rows = sum((min(l // 160, dims.n_audio_ctx - 10) + 10 - 1) // 2 + 1 for l in window_lens)
    per_pos = L * 14 * d * d * wbytes + L * 2 * T_rows * d * kvb
    self_kv = sum(L * 2 * (t + 1) * d * kvb * R for t in range(n_pos))
    return per_pos * n_pos + steps * V * d * wbytes + self_kv


def dram_traffic(model: str, kv: str, rows: int, dec: int):
    """DRAM bytes per decoder position of the dominant kernel from a COMMITTED ncu --set full capture
    (profiles/dram_traffic.json, keyed by workload), or None when no capture of this exact workload exists."""
    p = ROOT / "profiles" / "dram_traffic.json"
    if not p.exists():
        return None, None
    ent = json.loads(p.read_text()).get(f"{model}:{kv}:{rows}rows:dec{dec}")
    return (ent["dram_bytes_per_position"], ent["source"]) if ent else (None, None)


def run_config(args, cfg, ctx):
    """One workload: build the model + session, time the device path and the end-to-end path, profile the decoder launch."""
    import torch
    import torch.distributed as dist
    from whisper_burn_b200 import audio, ffi, model, shard, synth, transcribe
    model_name, chunks_per_gpu, kv = cfg
    world, rank, local_rank, dev = ctx["world"], ctx["rank"], ctx["local_rank"], ctx["dev"]
    dims, w_np = synth.make_weights(model_name, seed=0)
    sp = synth.special_tokens(dims)
    chunk_ids = [rank * chunks_per_gpu + i for i in range(chunks_per_gpu)]
    chunks = [synth.chunk_waveform(c, CHUNK_SAMPLES) for c in chunk_ids]
    is_special = (np.arange(dims.n_vocab) >= sp.first_special).astype(np.uint8)
    key = model_name
    if key not in ctx["models"]:
        ctx["models"].clear()          # one model resident at a time
        ctx["models"][key] = (model.Whisper(dims, w_np, device=local_rank), w_np if (rank == 0 and world == 1) else None)
    wh, w_keep = ctx["models"][key]
    window_len = audio.max_waveform_samples(dims.n_audio_ctx - 10)        # transcribe.rs:32-34 (C ABI, host side)
    bounds = transcribe.window_bounds(CHUNK_SAMPLES, 16000, window_len)   # transcribe.rs:114-138
    n_win = len(bounds) * len(chunks)
    sess = transcribe.Session(wh, max_windows=n_win, max_beams=max(args.beam, 1), max_text_len=4 + args.max_depth + 1,
                              kv_dtype=ffi.WB_KV_F16 if kv == "f16" else ffi.WB_KV_F32)

    # ---- inputs resident in HBM (value) and in pinned host memory (e2e)
    flat = np.concatenate(chunks)
    wave_dev = torch.from_numpy(flat).to(dev)
    offsets = [ci * CHUNK_SAMPLES + s for ci in range(len(chunks)) for (s, e) in bounds]
    lens = [e - s for _ in range(len(chunks)) for (s, e) in bounds]
    wave_pinned = torch.from_numpy(flat).pin_memory()
    pinned_np = wave_pinned.numpy()
    flush_buf = ctx["flush"]

    total_units = world * len(chunks)
    cap = 4 + args.max_depth + 1
    gather = shard.TokenGather(world * n_win, cap, dev) if world > 1 else None
    gather_e2e = shard.TokenGather(total_units, cap * 4, dev) if world > 1 else None

    def step_device():
        toks = sess.transcribe_windows_dev(wave_dev.data_ptr(), offsets, lens, sp, is_special, args.beam, args.max_depth)
        if gather is not None:   # the one exchange step: final token gather over NCCL/NVLink
            gather(toks)
        return toks

    def step_e2e():
        out = sess.waveforms_to_tokens([pinned_np[ci * CHUNK_SAMPLES:(ci + 1) * CHUNK_SAMPLES] for ci in range(len(chunks))],
                                       sp, is_special, 16000, args.beam, args.max_depth)
        if gather_e2e is not None:
            gather_e2e(out)
        return out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
        step_e2e()
    # the cyclic collector stays off inside the timed regions: a collection over the weight dictionaries costs milliseconds on a
    # 10 ms step (the 8-GPU run of round 2 had one 14 ms step among 10.7 ms ones; host-side noise of this kind, cause not isolated)
    import gc
    gc.collect()
    gc.disable()
    # ---- timed region: device path
    barrier()
    ffi.lib().wb_kernel_launch_count_reset()
    dev_ms, wall_ms, phase = [], [], {"logmel": 0.0, "encoder": 0.0, "decode": 0.0}
    toks = None
    for _ in range(args.steps):
        flush_buf.fill_(1)              # flush L2 between timed iterations
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        toks = step_device()
        torch.cuda.synchronize()
        wall_ms.append(1000.0 * (time.perf_counter() - t0))
        t = sess.last_timings_ms()      # CUDA events on the library's stream
        dev_ms.append(t["total"])
        for k in phase:
            phase[k] += t[k] / args.steps
    launches = int(ffi.lib().wb_kernel_launch_count())
    barrier()
    # ---- timed region: end to end through the user-facing call, host buffers
    e2e_ms = []
    for _ in range(args.steps):
        flush_buf.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        merged = step_e2e()
        torch.cuda.synchronize()
        e2e_ms.append(1000.0 * (time.perf_counter() - t0))
    barrier()
    gc.enable()
    steps_run = sess.last_steps()
    outputs = None
    if args.dump_outputs and rank == 0:   # what each timed path returned in its last step, every rank's units in global order
        outputs = {"window_tokens": gather.as_lists(gather.np_out) if gather is not None else toks,
                   "chunk_tokens": gather_e2e.as_lists(gather_e2e.np_out) if gather_e2e is not None else merged}

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    per_rank = None
    if world > 1:   # per-rank step times (the scaling loss is launch skew + the all-gather, see DESIGN.md section 8)
        t = torch.tensor([float(np.mean(wall_ms)), float(np.mean(dev_ms))], dtype=torch.float64, device=dev)
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = [[round(float(x[0]), 3), round(float(x[1]), 3)] for x in allt]
    ms_step = max_over_ranks(float(np.mean(wall_ms)))
    ms_dev = max_over_ranks(float(np.mean(dev_ms)))
    ms_e2e = max_over_ranks(float(np.mean(e2e_ms)))
    audio_s = CHUNK_SECONDS * total_units
    value = audio_s / (ms_step / 1000.0)
    e2e_val = audio_s / (ms_e2e / 1000.0)

    # ---- roofline of the dominant kernel: the persistent decoder (ONE launch = prompt prefill + all greedy steps).
    # Algorithmic bytes per position, SURVEY.md 8d: decoder weights ONCE per step for the whole batch `(L*14*d^2 + V*d) * 2`
    # (the vocabulary matrix only on positions that produce logits), every window's cross K/V `L*2*T*d*kvb`, every row's self
    # K/V up to the current position.  Re-reads a kernel's decomposition forces (e.g. one weight stream per row cluster served
    # by L2) are NOT algorithmic bytes; they are reported as `l2_weight_streams`.
    hbm_peak, peak_src = peaks()
    roof = None
    if rank == 0:
        R = n_win
        prof_steps = args.max_depth
        n_pos = prof_steps + 3
        alg_bytes = algorithmic_bytes(dims, lens, 2 if wh.weights_fp16_exact else 4, 2 if kv == "f16" else 4, prof_steps)
        try:
            k_ms, _ = sess.profile_decode(sp, prof_steps)          # per-position average of one timed launch (CUDA events, library stream)
            launch_ms = k_ms * n_pos
            ach = alg_bytes / (launch_ms * 1e-3) / 1e9
            dec = sess.last_decoder()
            per_pos_traffic, src = dram_traffic(model_name, kv, R, dec)
            names = {3: "dec3_kernel (persistent grid-barrier FMA decoder, decoder3.cu)",
                     4: "dec4_kernel (persistent cluster/DSMEM decoder, decoder4.cu)",
                     5: "dec5_kernel (persistent batched tensor-core decoder, decoder5.cu)",
                     6: "dec6_kernel (persistent head-fused cluster decoder, decoder6.cu)"}
            roof = {"bound": "hbm", "kernel": names.get(dec, f"dec{dec}_kernel") + f"; one launch = {n_pos} positions",
                    "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "traffic": per_pos_traffic * n_pos if per_pos_traffic else None, "traffic_source": src,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": int(alg_bytes), "ms_per_launch": launch_ms,
                    "us_per_position": k_ms * 1e3, "positions_per_launch": n_pos,
                    "l2_weight_streams": R if dec in (4, 6) else 1,
                    "note": "algorithmic bytes per SURVEY.md 8d (weights once per position for the whole batch); "
                            "l2_weight_streams = how many times the kernel's decomposition streams the layer weights per position "
                            "(served by L2 for models that fit it)"}
        except Exception as ex:   # noqa: BLE001
            roof = {"bound": "hbm", "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None, "traffic": None,
                    "error": str(ex)}

    res = None
    if rank == 0:
        h2d = int(sum(lens)) * 4
        d2h = int(n_win * (cap + 1) * 4 + 4)
        res = {
            "workload": workload_name(model_name, len(chunks), args.beam, args.max_depth), "model": model_name,
            "chunks_per_gpu": len(chunks), "kv_cache": kv, "windows_per_gpu": n_win,
            "value": value, "unit": "audio-s/s", "ms_per_step": ms_step, "device_ms_per_step": ms_dev, "phase_ms": phase,
            "rtf": (ms_step / 1000.0) / audio_s, "decode_steps_executed": steps_run,
            "e2e": {"value": e2e_val, "unit": "audio-s/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e, "api": "wb_waveforms_to_tokens (windowing + batched decode + overlap merge), pinned host waveforms"},
            "gpu_launches": launches // args.steps, "roofline": roof,
            "wall_ms_each": [round(v, 3) for v in wall_ms], "e2e_ms_each": [round(v, 3) for v in e2e_ms],
            "weights": "fp16-exact synthetic (tensor-core path)" if wh.weights_fp16_exact else "not fp16-exact: fp32 SIMT path",
            "tokens_checksum": int(sum(sum(t) for t in toks) % (1 << 31)),
        }
        if per_rank is not None:
            res["per_rank_ms_wall_dev"] = per_rank
    sess.close()
    return res, (dims, w_keep, sp, chunks[0], chunk_ids[0]), outputs


def write_outputs(out_dir, outputs: dict) -> None:
    """One DIR/<name>.npy per token id list of lists: float64 [n, longest list], padded with -1."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, lists in outputs.items():
        m = np.full((len(lists), max((len(t) for t in lists), default=0)), -1.0)
        for i, t in enumerate(lists):
            m[i, :len(t)] = t
        np.save(d / f"{name}.npy", m)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import wb200  # noqa: F401

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    ctx = {"world": world, "rank": rank, "local_rank": local_rank, "dev": dev, "models": {},
           "flush": torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)}   # > 126 MB L2

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    results, head_inputs, dumps = [], None, {}
    for i, cfg in enumerate(args.config_list):
        res, inputs, outputs = run_config(args, cfg, ctx)
        results.append(res)
        if i == 0:
            head_inputs = inputs
        if outputs is not None:
            dumps.update({f"{i}_{cfg[0]}_{cfg[1]}chunks_{cfg[2]}_{k}": v for k, v in outputs.items()})
    clocks = sampler.stop() if sampler else None
    if dumps:
        write_outputs(args.dump_outputs, dumps)

    # ---- CPU baseline beside the headline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import synth as o_synth
        dims, w_np, sp, chunk0, cid = head_inputs
        if w_np is None:
            from whisper_burn_b200 import synth
            _, w_np = synth.make_weights(args.config_list[0][0], seed=0)
        torch.set_num_threads(host_cores())
        w_t = o_synth.to_torch(w_np)
        span, dt, nw, _ = cpu_reference_pass(args.beam, args.max_depth, dims, w_t, sp, chunk0, args.cpu_baseline_windows)
        cpu = {"value": span / dt, "unit": "audio-s/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"{nw} of 3 reference windows of chunk {cid} ({span:.2f} s audio), greedy depth {args.max_depth}, "
                         f"oracle reference-cost mode (no KV cache), {dt:.2f} s CPU"}

    if rank == 0:
        h = results[0]
        line = {
            "metric": "audio-seconds/sec", "value": h["value"], "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": h["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (fp16-exact weights, fp32 activations/accumulate)", "data": "synthetic",
            "config": {"workload": h["workload"],
                       "parallelism": f"dp{world} (windows sharded, weights replicated, one NCCL token all-gather)",
                       "l2": "flushed between timed iterations (256 MB write)", "timing": "wall clock around the synchronous C-ABI call, "
                       "torch.cuda.synchronize() both sides; device_ms = CUDA events on the library stream",
                       "decode_steps_executed": h["decode_steps_executed"], "windows_per_gpu": h["windows_per_gpu"], "kv_cache": h["kv_cache"]},
            "device_ms_per_step": h["device_ms_per_step"], "phase_ms": h["phase_ms"], "rtf": h["rtf"],
            "e2e": h["e2e"], "gpu_launches": h["gpu_launches"], "clocks": clocks, "roofline": h["roofline"], "cpu_baseline": cpu,
            "tokens_checksum": h["tokens_checksum"],
            "configs": results,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """Exactly one JSON line on the real stdout (native libraries such as NCCL print banners to fd 1)."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)            # everything else that writes to fd 1 goes to stderr
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
