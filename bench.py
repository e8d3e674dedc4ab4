#!/usr/bin/env python
"""bench.py -- 44.1 kHz audio-seconds restored per wall-second (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W           (N>1: launched by torchrun, one rank/GPU)
  python bench.py --impl reference ...                    (the reference's CPU path: oracle port)

One step = one pass of the restore() hot path (vfx_restore: STFT+mel -> denoiser+UNet -> vocoder -> trim) over a batch
of synthetic degraded utterances.  N = 1: BASELINE configs[2], 32 x 10 s, mode 0.  N > 1: configs[3]'s per-GPU share,
64 x 10 s per GPU (512 x 10 s over 8 GPUs), weak scaling; the N = 1 line carries the 64-item rate under
`workloads.batch64_1gpu` as the consistent single-GPU base.

  value   device-resident whole-job throughput (CUDA-graph replay; at N > 1 including the NCCL gather of the waveforms
          to rank 0, issued on a side stream so that it overlaps the next step's compute)
  e2e     N = 1: the public API call, VoiceFixer.restore_batch (numpy in -> numpy out, pinned host memory): H2D of the
          step's inputs, the launch sequence, D2H of the waveforms, every step.  N > 1: per rank H2D of its shard ->
          launch sequence -> NCCL gather -> rank 0 copies the WHOLE gathered result to its host.
  dtype   the headline runs at the reference CUDA path's arithmetic class, tf32 (cuDNN TF32 convolutions, SURVEY D10);
          the fp16 mode (tf32's 10-bit mantissa in 2-byte operands: tf32's parity at bf16's speed, within fp16's exponent
          range) and the bf16 mode are measured in the same run and reported under `modes`, each with its own parity.

The N = 1 line also carries: `roofline` (ResStack pair unit of SURVEY 8d), `cpu_baseline` (oracle port on the host cores,
bounded sample), `parity` (waveform error of each precision against that oracle output; out of tolerance FAILS the run),
`workloads` (configs[1] vocoder-only latency, configs[4] 10 min long-form through VoiceFixer.restore_inmem in modes
0/1/2, the 64-item batch) and `gpu_library_baseline` (the reference's op sequence through stock PyTorch on the same GPU).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = "audio_sec_restored_per_wall_sec_44k1"
UNIT = "audio-s/s"
FLOP_PER_AUDIO_SEC = 118.44e9        # BASELINE.md §2: 1184.4 GFLOP per 10 s utterance


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def host_threads():
    """Usable host threads: affinity mask and cgroup quota, not just os.cpu_count()."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


_BEST_THREADS = None


def best_cpu_threads():
    """PyTorch CPU throughput of this path peaks well below a 128-thread box's core count (small
    GEMMs + a 4000-step GRU loop oversubscribe); calibrate on 0.3 s of audio and keep the fastest."""
    global _BEST_THREADS
    if _BEST_THREADS is None:
        from voicefixer_b200 import synthetic
        from oracle import vf_oracle as O
        ana, voc = synthetic.make_analysis_state(0), synthetic.make_vocoder_state(1)
        wav = synthetic.make_utterances(1, seconds=0.3, seed=5)[0]
        n = host_threads()
        best = None
        for t in sorted({min(n, c) for c in (8, 16, 32, 64, n)}):
            torch.set_num_threads(t)
            O.restore_inmem(wav, ana, voc, mode=0)
            t0 = time.perf_counter()
            O.restore_inmem(wav, ana, voc, mode=0)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, t)
            if dt > 20:
                break
        _BEST_THREADS = best[1]
    return _BEST_THREADS


def cpu_reference_rate(seconds, threads=None):
    """The reference's CPU path (oracle port of restore_inmem, PyTorch fp32) on the host cores."""
    from voicefixer_b200 import synthetic
    from oracle import vf_oracle as O
    threads = threads or best_cpu_threads()
    torch.set_num_threads(threads)
    ana, voc = synthetic.make_analysis_state(0), synthetic.make_vocoder_state(1)
    wav = synthetic.make_utterances(1, seconds=seconds, seed=1234)[0]

    def run():
        t0 = time.perf_counter()
        run.out = O.restore_inmem(wav, ana, voc, mode=0)                  # kept: the checker for the parity figure
        return time.perf_counter() - t0
    run.wav = wav
    return run, threads


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; the
    reference is pure Python and cannot be installed offline with its missing dependencies)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.steps + args.warmup
    run1, threads = cpu_reference_rate(1.0)
    t1 = run1()                                                  # calibration, ~1 s of audio
    seconds = float(min(10.0, max(1.0, 150.0 / max(n, 1) / max(t1, 1e-3))))
    run, threads = cpu_reference_rate(seconds)
    for _ in range(args.warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run()
    dt = (time.perf_counter() - t0) / args.steps
    v = seconds / dt
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{'configs[2]' if args.gpus == 1 else 'configs[3]'}: batch {args.batch} x {args.seconds:g} s synthetic degraded "
                               f"44.1 kHz mono utterances per GPU, mode 0, seeded synthetic checkpoints (bounded sample per step: "
                               f"1 x {seconds:.1f} s utterance)",
                   "impl": "oracle port of voicefixer/base.py:106-139 (PyTorch fp32 on the host cores)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} x 1 x {seconds:.1f} s utterance"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))



TOL = {"tf32": (2e-3, 1e-3), "fp16": (2e-3, 1e-3), "bf16": (3e-2, 5e-3), "fp32": (2e-4, 1e-4)}      # (rel-RMS, mean-abs) vs the oracle, tests/test_parity_gpu.py
DTYPE = {"bf16": "bf16", "tf32": "tf32", "fp32": "f32", "fp16": "f16"}


def wl_longform(vf, steps=2, modes=(0, 1, 2)):
    """configs[4]: ONE 10-minute utterance through the public entry point VoiceFixer.restore_inmem (numpy -> numpy,
    voicefixer/base.py:106-139: twenty independent 30 s segments, batched), every mode; plus the latency to the first
    restored 30 s segment when the caller asks for segment 0 alone."""
    from voicefixer_b200 import synthetic
    base = synthetic.make_utterances(1, seconds=30.0, seed=77)[0]
    wav = np.tile(base, 20)                                           # 600 s
    out = {"workload": "configs[4]: 1 x 10 min utterance = 20 x 30 s segments (T = 3001 frames each) through "
                       "VoiceFixer.restore_inmem, host numpy in -> host numpy out, 1 GPU", "ms_per_mode": {}}
    for mode in modes:
        try:
            torch.manual_seed(mode)
            vf.restore_inmem(wav, cuda=True, mode=mode)               # warm-up (workspace allocation)
            t0 = time.perf_counter()
            for _ in range(steps):
                y = vf.restore_inmem(wav, cuda=True, mode=mode)
            dt = (time.perf_counter() - t0) / steps
            out["ms_per_mode"][str(mode)] = dt * 1e3
            if mode == 0:
                out.update({"value": 600.0 / dt, "unit": UNIT, "latency_to_full_waveform_ms": dt * 1e3,
                            "finite": bool(np.isfinite(y).all()), "out_shape": list(y.shape)})
        except Exception as e:
            out["ms_per_mode"][str(mode)] = f"{type(e).__name__}: {e}"
    try:
        vf.restore_inmem(base, cuda=True, mode=0)
        t1 = time.perf_counter()
        vf.restore_inmem(base, cuda=True, mode=0)
        out["latency_to_first_segment_ms"] = (time.perf_counter() - t1) * 1e3
    except Exception as e:
        out["latency_to_first_segment_ms"] = f"{type(e).__name__}: {e}"
    return out


def wl_vocoder(vf, steps=10):
    """configs[1]: the synthesis-only path, Vocoder.forward (vocoder/base.py:42-56) on ONE 10 s utterance's linear 128-bin
    mel [1, 1, 1001, 128] -> waveform [1, 1, 443646]: batch-1 latency.  Device-resident (CUDA events, median) and through
    the public call with a host tensor in / host tensor out."""
    from voicefixer_b200 import synthetic
    eng = vf._engine
    wav = torch.from_numpy(synthetic.make_utterances(1, seconds=10.0, seed=1234)).cuda()
    mel = eng.frontend(wav)
    host_mel = mel.cpu()[:, None]                                     # (1, 1, 1001, 128) as the reference API takes it
    for _ in range(3):
        eng.vocoder(mel)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        eng.vocoder(mel)
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(steps))[steps // 2]
    vf._model.vocoder(host_mel, cuda=False)
    t0 = time.perf_counter()
    for _ in range(steps):
        y = vf._model.vocoder(host_mel, cuda=False)                   # host in -> host out
    ms_api = (time.perf_counter() - t0) / steps * 1e3
    return {"workload": "configs[1]: Vocoder.forward on 1 x 10 s linear 128-bin mel (1001 frames -> 443646 samples), batch 1",
            "value": 10.0 / (ms * 1e-3), "unit": UNIT, "ms_per_call_device": ms,
            "api_host_to_host": {"value": 10.0 / (ms_api * 1e-3), "ms_per_call": ms_api, "out_shape": list(y.shape)}}


def wl_stream(vf, seconds=12.0, chunk=1.0, ctx=0.5):
    """SURVEY 8f-3 streaming path: VoiceFixer.restore_stream fed 0.1 s blocks; per-window compute time (host -> host, B = 1)
    and the resulting time to the first restored audio = (chunk + context) seconds of arrival + one window's compute."""
    from voicefixer_b200 import synthetic
    wav = synthetic.make_utterances(1, seconds=seconds, seed=91)[0]
    blocks = [wav[i:i + 4410] for i in range(0, len(wav), 4410)]
    list(vf.restore_stream(blocks[:40], chunk_seconds=chunk, context_seconds=ctx))          # warm-up (workspace, lazy init)
    gaps, n, t_prev = [], 0, time.perf_counter()
    for y in vf.restore_stream(blocks, chunk_seconds=chunk, context_seconds=ctx):
        t = time.perf_counter()
        gaps.append((t - t_prev) * 1e3); t_prev = t; n += len(y)
    steady = sorted(gaps[1:-1])[len(gaps[1:-1]) // 2] if len(gaps) > 2 else gaps[0]
    return {"workload": f"restore_stream: {seconds:g} s fed in 0.1 s blocks, chunk {chunk:g} s + {ctx:g} s context each side (B = 1 windows)",
            "compute_ms_per_window": steady, "first_window_compute_ms": gaps[0],
            "time_to_first_audio_ms": (chunk + ctx) * 1e3 + gaps[0], "real_time_factor": chunk * 1e3 / steady,
            "samples_out": n, "samples_in": int(len(wav))}


def wl_cli(precision, n_files=8, seconds=10.0):
    """SURVEY 8f-1: the CLI `python -m voicefixer_b200 --infolder .. --outfolder ..` (mirror of voicefixer/__main__.py) on a
    folder of wav files: disk -> decode -> GPU -> encode -> disk, checkpoints read from ~/.cache/voicefixer like the reference.
    Wall time of main() includes the one-off checkpoint load; `jobs_wall_s` is the pipeline alone."""
    import contextlib, io, re, tempfile
    from voicefixer_b200 import synthetic, wavio
    from voicefixer_b200.__main__ import main as cli_main
    old_home, old_prec = os.environ.get("HOME"), os.environ.get("VFX_PRECISION")
    with tempfile.TemporaryDirectory() as td:
        try:
            os.environ["HOME"], os.environ["VFX_PRECISION"] = td, precision
            synthetic.write_checkpoints(td, seed=0)
            src, dst = os.path.join(td, "in"), os.path.join(td, "out")
            os.makedirs(src)
            wavs = synthetic.make_utterances(n_files, seconds=seconds, seed=95)
            for i, w in enumerate(wavs):
                wavio.save_wave(w[None], os.path.join(src, f"u{i:02d}.wav"))
            buf = io.StringIO()
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(buf):
                rc = cli_main(["--infolder", src, "--outfolder", dst])
            wall = time.perf_counter() - t0
            m = re.search(r"Done: (\d+) job\(s\) in ([0-9.]+) s", buf.getvalue())
            jobs_wall = float(m.group(2)) if m else None
            ok = rc == 0 and len(os.listdir(dst)) == n_files
        finally:
            if old_home is None: os.environ.pop("HOME", None)
            else: os.environ["HOME"] = old_home
            if old_prec is None: os.environ.pop("VFX_PRECISION", None)
            else: os.environ["VFX_PRECISION"] = old_prec
    return {"workload": f"CLI folder mode: {n_files} x {seconds:g} s wav files, disk -> GPU -> disk, one utterance per launch sequence "
                        "(reference semantics), reader / writer threads", "ok": ok, "wall_s_including_checkpoint_load": wall,
            "jobs_wall_s": jobs_wall, "value": (n_files * seconds / jobs_wall) if jobs_wall else None, "unit": UNIT}


def csrc_sha(files=None):
    """Hash of CUDA sources (all of csrc/, or the listed files): an ncu traffic figure is only quoted when the kernel it was
    captured from is built from the same sources as the one that just ran."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "voicefixer_b200", "csrc")
    for f in sorted(files or os.listdir(d)):
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def roofline_from(rep, B, L_by_stack, precision, peaks, peaks_src, tot_ms):
    """SURVEY 8(d): the unit of the HBM-bound ResStack kernels is the PAIR -- read x once, write x' once,
    2 * C * L * 4 bytes per item -- whether a pair is one fused launch or two.  `frac` uses that; the kernel-level
    figures on the builder's own per-launch byte model (DESIGN.md 4) go under `other`."""
    cands = []
    for j, C in ((3, 64), (2, 128), (1, 256), (0, 512)):
        fused = rep.get(f"voc.rs{j}.pair")
        c1, c2 = rep.get(f"voc.rs{j}.c1"), rep.get(f"voc.rs{j}.c2")
        if fused:
            ms_pair, n = fused["ms"] / fused["count"], fused["count"]
            kname = ("resstack_pair3_kernel (one SM, residual stashed in TMEM)" if precision == "tf32" and C == 64
                     else "resstack_pair_kernel" if C == 64 else "resstack_pair2_kernel (two-CTA cluster)")
            kern = f"{kname} [voc.rs{j}.pair]"
            flops, model_bytes = fused["flops"] / fused["count"], fused["bytes"] / fused["count"]
        elif c1 and c2:
            ms_pair, n = (c1["ms"] + c2["ms"]) / c2["count"], c2["count"]
            kern = (f"conv_ts_kernel (weights in TMEM) + conv_gemm_tc_kernel for large dilations [voc.rs{j}.c1 + voc.rs{j}.c2]"
                    if precision == "tf32" and C == 128 else f"conv_gemm_tc_kernel x2 [voc.rs{j}.c1 + voc.rs{j}.c2]")
            flops = (c1["flops"] + c2["flops"]) / c2["count"]
            model_bytes = (c1["bytes"] + c2["bytes"]) / c2["count"]
        else:
            continue
        cands.append(dict(j=j, C=C, ms_pair=ms_pair, n=n, kern=kern, flops=flops, model_bytes=model_bytes,
                          pair_bytes=2.0 * C * L_by_stack[j] * 4.0 * B, total_ms=ms_pair * n))
    tc_peak = peaks["bf16_tflops_sustained"] * (0.5 if precision == "tf32" else 1.0)      # tf32 runs at half the bf16 rate
    ridge = tc_peak * 1e3 / peaks["hbm_gbs"]
    hbm = [c for c in cands if c["flops"] / c["pair_bytes"] < ridge]
    dom = max(hbm or cands, key=lambda c: c["total_ms"])
    gbs = dom["pair_bytes"] / (dom["ms_pair"] * 1e-3) / 1e9
    tf = dom["flops"] / (dom["ms_pair"] * 1e-3) / 1e12
    traffic, tnote = None, "no ncu capture of these sources committed"
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        ent = tj.get(f"{'bf16' if precision == 'fp16' else precision}:voc.rs{dom['j']}.pair:B{B}")       # fp16 moves bf16's bytes
        if ent and ent.get("csrc_sha") == csrc_sha(ent.get("files")):
            traffic, tnote = ent["dram_bytes_per_pair"], ent.get("source", "profiles/")
        elif ent:
            tnote = "capture in profiles/ncu_traffic.json is from older sources: not quoted"
    return {"bound": "hbm", "kernel": dom["kern"], "unit_of_work": f"ResStack pair, C = {dom['C']}, {B} x {L_by_stack[dom['j']]} positions",
            "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
            "traffic": traffic, "traffic_note": tnote, "peak_source": f"{peaks_src} (hbm_gbs)",
            "algorithmic_bytes_per_pair": dom["pair_bytes"], "algorithmic_flops_per_pair": dom["flops"],
            "pairs_in_step": dom["n"], "avg_pair_ms": dom["ms_pair"], "share_of_step": dom["total_ms"] / tot_ms,
            "other": {"builder_byte_model_gbs": dom["model_bytes"] / (dom["ms_pair"] * 1e-3) / 1e9,
                      "builder_byte_model_frac": dom["model_bytes"] / (dom["ms_pair"] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                      "tflops": tf, "tensor_peak_tflops": tc_peak, "flop_per_byte": dom["flops"] / dom["pair_bytes"], "ridge": ridge,
                      "all_stacks": {f"rs{c['j']} (C={c['C']})": {"pair_ms": round(c["ms_pair"], 4),
                                                                  "pair_gbs": round(c["pair_bytes"] / (c["ms_pair"] * 1e-3) / 1e9, 1),
                                                                  "tflops": round(c["flops"] / (c["ms_pair"] * 1e-3) / 1e12, 1)} for c in cands}}}


DUMP_LIMIT = 64 * 10 ** 6           # bytes --dump-outputs writes at most


def dump_outputs(out_dir, waveforms):
    """--dump-outputs: the (utterances, samples) float32 waveforms a caller of the timed path receives, from its last
    step, as waveforms.npy.  Above DUMP_LIMIT: a fixed seeded sample of the flattened array, with the flat indices it
    took (ascending) in waveforms_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    y = waveforms.float().cpu().numpy()
    if y.nbytes > DUMP_LIMIT:
        n = (DUMP_LIMIT - 4096) // (y.itemsize + 8)                     # 4096: room for the two .npy headers
        idx = np.sort(np.random.default_rng(0).choice(y.size, n, replace=False))
        np.save(os.path.join(out_dir, "waveforms_index.npy"), idx.astype(np.float64))
        y = y.reshape(-1)[idx]
    np.save(os.path.join(out_dir, "waveforms.npy"), y)


def measure_batch(args, precision, rank, world, local, B, full=True):
    """One engine at `precision`: resident and end-to-end throughput of the batch step (see the module docstring)."""
    import torch.distributed as dist
    from voicefixer_b200 import parallel, synthetic, api
    from voicefixer_b200.engine import Engine
    from voicefixer_b200.weights import pack_analysis, pack_vocoder
    dev = f"cuda:{local}"
    eng = Engine(device=local, precision=precision)
    if rank == 0:
        packed = {}
        packed.update(pack_analysis(synthetic.make_analysis_state(0), precision))
        packed.update(pack_vocoder(synthetic.make_vocoder_state(1), precision))
        eng.upload(packed)
        table, arena = eng.table, eng.arena
    else:
        table, arena = None, None
    torch.cuda.synchronize()
    t_b0 = time.perf_counter()
    table, arena = parallel.broadcast_arena(table, arena, dev)          # collective 1 of 2: once, start-up
    torch.cuda.synchronize()
    bcast_ms = (time.perf_counter() - t_b0) * 1e3
    if rank != 0:
        eng.attach(arena, table)
    vf = api.VoiceFixer.from_engine(eng)

    L = int(round(args.seconds * 44100))
    distinct = synthetic.make_utterances(min(B, 8), seconds=args.seconds, seed=1234 + rank)
    host_in = vf.pinned_empty((B, L))
    host_in[...] = np.concatenate([distinct] * ((B + len(distinct) - 1) // len(distinct)))[:B]
    host_out = vf.pinned_empty((B, L))
    dev_in = torch.from_numpy(host_in).to(dev)
    dev_out = torch.empty(B, L, device=dev)
    ws_gb = eng.workspace_bytes(B, L) / 1e9
    main = torch.cuda.current_stream()
    graph = None
    if not args.no_graph:
        graph = eng.make_graph(dev_in, dev_out, mode=0)

    def run_restore():
        if graph is not None:
            graph.replay()
        else:
            eng.restore(dev_in, mode=0, out=dev_out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- N > 1: collective 2 of 2, the waveform gather, on a side stream (overlaps the next step's compute)
    gplan = comm = None
    if world > 1:
        gplan = parallel.WaveformGather(B, L, torch.float32, dev)       # shard sizes exchanged here, once
        comm = torch.cuda.Stream(device=dev)
        gsrc = [torch.empty(B, L, device=dev) for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        ev_ready = torch.cuda.Event()
        host_full = torch.empty(world * B, L).pin_memory() if rank == 0 else None
    counter = [0]
    gathered = [None]

    def step(e2e):
        k = counter[0] & 1
        counter[0] += 1
        if world == 1:
            if e2e:
                vf.restore_batch(host_in, out=host_out)                 # the public call: numpy in -> numpy out
            else:
                run_restore()
            return
        if e2e:
            dev_in.copy_(torch.from_numpy(host_in), non_blocking=True)
        run_restore()
        main.wait_event(ev_done[k])                                     # the gather that last read gsrc[k] has finished
        gsrc[k].copy_(dev_out, non_blocking=True)
        ev_ready.record(main)
        with torch.cuda.stream(comm):
            comm.wait_event(ev_ready)
            y = gathered[0] = gplan(gsrc[k])
            if e2e and rank == 0:
                host_full.copy_(y, non_blocking=True)                   # rank 0 reads back the WHOLE gathered result
            ev_done[k].record(comm)

    def timed(e2e, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for _ in range(steps):
            step(e2e)
        if comm is not None:
            main.wait_stream(comm)
        e1.record(main)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)                   # timing plumbing, outside the timed region
        return float(ms.item())

    for _ in range(args.warmup):
        step(False)
    sampler = ClockSampler(local)
    if rank == 0 and full:
        sampler.start()
    ms_step = timed(False, args.steps) / args.steps
    clocks = sampler.stop() if rank == 0 and full else None
    if rank == 0 and full and args.dump_outputs:
        dump_outputs(args.dump_outputs, dev_out if world == 1 else gathered[0])
    l0 = eng.launch_count(); eng.restore(dev_in, mode=0, out=dev_out); torch.cuda.synchronize()
    launches = (eng.launch_count() - l0) * args.steps                  # graph replays bypass the library's counter
    audio_per_step = world * B * args.seconds
    res = {"value": audio_per_step / (ms_step / 1e3), "ms_per_step": ms_step, "gpu_launches": launches, "clocks": clocks,
           "ws_gb": ws_gb, "bcast_ms": bcast_ms, "graph": graph is not None}
    step(True)
    ms_e2e = timed(True, args.steps) / args.steps
    res["e2e"] = {"value": audio_per_step / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e,
                  "h2d_bytes_per_step": world * B * L * 4, "d2h_bytes_per_step": world * B * L * 4,
                  "path": "VoiceFixer.restore_batch(numpy (B, L) pinned) -> numpy (B, L): H2D + CUDA-graph replay + D2H per call"
                          if world == 1 else
                          "per rank: pinned H2D of its shard -> CUDA-graph replay -> NCCL gather to rank 0 (side stream) -> "
                          "rank 0 D2H of the whole gathered (N*B, L) result"}
    # ---- per-launch-group CUDA-event profile of one more step (same stream)
    eng.profile(True)
    eng.restore(dev_in, mode=0, out=dev_out)
    rep = eng.profile_report()
    eng.profile(False)
    res["rep"] = rep
    res["breakdown_ms"] = {t: round(r["ms"], 3) for t, r in sorted(rep.items(), key=lambda kv: -kv[1]["ms"])}
    res["vf"], res["eng"] = vf, eng
    return res


def parity_of(eng, wav, ref, precision):
    y = eng.restore(torch.from_numpy(wav)[None].to(f"cuda:{eng.device}")).cpu().numpy().astype(np.float64)
    ref = np.asarray(ref, dtype=np.float64).reshape(y.shape)
    err = float(np.sqrt(np.mean((y - ref) ** 2)))
    rms = float(np.sqrt(np.mean(ref ** 2)))
    tol_rms, tol_mae = TOL[precision]
    mae = float(np.mean(np.abs(y - ref)))
    return {"wav_rms_err": err, "wav_rms_ref": rms, "rel_rms": err / rms, "mean_abs_err": mae,
            "tolerance": {"rel_rms": tol_rms, "mean_abs": tol_mae}, "ok": bool(err / rms < tol_rms and mae < tol_mae)}

def torch_gpu_result(args, B):
    """Library baseline: the reference's op sequence (oracle restatement: F.conv1d/conv2d/conv_transpose, batch_norm,
    matmul-based GRU loop) executed by stock PyTorch on cuda:0 with its defaults (TF32 convolutions through cuDNN).
    Reported for context only; none of this repo's kernels run here."""
    from voicefixer_b200 import synthetic
    from oracle import vf_oracle as O
    dev = "cuda:0"
    # fp32 NCHW activations of the reference layout: ~3 GB per 10 s item at the peak
    ana = {k: v.to(dev) for k, v in synthetic.make_analysis_state(0).items()}
    voc = {k: v.to(dev) for k, v in synthetic.make_vocoder_state(1).items()}
    O.mel_weight = (lambda f: (lambda: f().to(dev)))(O.mel_weight)
    # the oracle's explicit Python GRU loop would be unfair to PyTorch: use cuDNN's nn.GRU like the reference does
    grus = {}
    for g in ("7", "8"):
        m = torch.nn.GRU(512, 256, num_layers=2, bidirectional=True, batch_first=True).to(dev)
        pre = f"generator.denoiser.{g}.gru."
        m.load_state_dict({k[len(pre):]: v for k, v in ana.items() if k.startswith(pre)})
        grus[f"generator.denoiser.{g}"] = m.eval()

    def bn_gru_cudnn(x, ana_, prefix, train):
        x = O._bn1(x, ana_, prefix + ".bn", train).squeeze(1)
        return grus[prefix](x)[0].unsqueeze(1)
    O.bn_gru = bn_gru_cudnn
    wav = torch.from_numpy(synthetic.make_utterances(min(B, 4), seconds=args.seconds, seed=1234)).repeat((B + 3) // 4, 1)[:B].to(dev)

    @torch.no_grad()
    def step():
        _, mel = O.frontend(wav, ana)
        out_mel = O.analysis(mel, ana)
        S = torch.abs(O.from_log(out_mel) / O.mel_weight()[None, None, None, :])
        S = 20 * torch.log10(torch.clamp(S, min=1e-5)) - 20.0
        S = torch.clip(8.0 * ((S + 115.0) / 115.0) - 4.0, -4.0, 4.0)[:, 0].transpose(1, 2)
        cond = torch.cat([S, torch.full((S.shape[0], 128, S.shape[-1] % 2 + 4), -4.0, device=dev)], -1)
        return O.trim_center(O.vocoder_generator(cond, voc), wav.shape[-1])

    for _ in range(max(1, min(args.warmup, 2))):
        step()
    torch.cuda.synchronize()
    steps = max(1, min(args.steps, 3))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    v = B * args.seconds / (ms * 1e-3)
    return ({"impl": "torch-gpu", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": 1, "steps": steps,
                      "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "dtype": "tf32/fp32 (torch defaults)",
                      "data": "synthetic",
                      "config": {"workload": f"batch {B} x {args.seconds:g} s, mode 0, PyTorch {torch.__version__} ops on cuda:0 "
                                             "(cuDNN convs/GRU, cuBLAS)", "note": "library baseline, context only"}})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch-gpu"],
                    help="b200: this repo; reference: the reference's CPU path (oracle port); torch-gpu: the same PyTorch "
                         "ops on the GPU through cuDNN/cuBLAS (library baseline, what the reference's cuda=True path runs)")
    ap.add_argument("--batch", type=int, default=0, help="utterances per GPU (default: 32 at N = 1 = configs[2]; 64 at N > 1 = configs[3]'s share)")
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--precision", default=os.environ.get("VFX_PRECISION", "tf32"),
                    help="tf32 (default: the reference CUDA path's arithmetic class), bf16, or fp32 (SIMT validation path)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the second precision mode, the workloads and the library baseline")
    ap.add_argument("--no-graph", action="store_true", help="launch the kernels of a step individually")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the waveforms of the last timed step to DIR/waveforms.npy (float32; over 64 MB, a fixed "
                         "seeded sample), to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        if not args.batch:
            args.batch = 32 if args.gpus == 1 else 64
        return run_reference(args)
    if args.impl == "torch-gpu":
        if not args.batch:
            args.batch = 32
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(torch_gpu_result(args, args.batch)))
        return
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    from voicefixer_b200 import parallel
    rank, world, local = parallel.init_from_env()
    assert world == args.gpus or world == 1, f"WORLD_SIZE {world} != --gpus {args.gpus}"
    torch.cuda.set_device(local)
    B = args.batch or (32 if world == 1 else 64)
    prec = args.precision
    peaks, peaks_src = measured_peaks()

    res = measure_batch(args, prec, rank, world, local, B)
    rep = res["rep"]
    tot_ms = sum(r["ms"] for r in rep.values())
    Tc = 1 + int(round(args.seconds * 44100)) // 441
    Tc = Tc + Tc % 2 + 4
    L_by_stack = {0: Tc * 7, 1: Tc * 49, 2: Tc * 147, 3: Tc * 441}
    roofline = roofline_from(rep, B, L_by_stack, prec, peaks, peaks_src, tot_ms)
    whole_tf = FLOP_PER_AUDIO_SEC * B * args.seconds / (res["ms_per_step"] * 1e-3) / 1e12
    roofline["whole_step"] = {"tflops": whole_tf, "frac_of_bf16_sustained": whole_tf / peaks["bf16_tflops_sustained"]}

    extras = rank == 0 and world == 1 and not args.no_extras
    cpu_baseline, parity, modes, workloads, lib_base = None, None, {}, {}, None
    run = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        run1, threads = cpu_reference_rate(1.0)
        t1 = run1()
        sample_s = float(min(10.0, max(1.0, round(20.0 / max(t1, 1e-3)))))      # ~20 s of CPU work
        run, threads = cpu_reference_rate(sample_s, threads)
        dt = run()
        cpu_baseline = {"value": sample_s / dt, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"1 x {sample_s:.0f} s utterance, restore_inmem mode 0 (oracle port, PyTorch fp32), "
                                  f"{dt:.1f} s wall, {threads} of {host_threads()} host threads (fastest of a sweep)"}
        # BASELINE metric, second half: waveform RMS vs the reference on identical input and weights.  The oracle output
        # of the baseline sample above is the checker (untimed, not in `value`); out of tolerance fails the run.
        parity = parity_of(res["eng"], run.wav, run.out, prec)
        parity["sample"] = f"the cpu_baseline utterance ({sample_s:.0f} s), oracle port vs this engine, same synthetic checkpoints"
    if extras:
        vf = res["vf"]
        try:
            workloads["vocoder"] = wl_vocoder(vf, steps=max(10, args.steps))
        except Exception as e:
            workloads["vocoder"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            workloads["longform"] = wl_longform(vf)
        except Exception as e:
            workloads["longform"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            workloads["stream"] = wl_stream(vf)
        except Exception as e:
            workloads["stream"] = {"error": f"{type(e).__name__}: {e}"}
    # free the headline engine before the next ones
    res.pop("vf"); res.pop("eng"); res.pop("rep")
    import gc
    gc.collect(); torch.cuda.empty_cache()
    if extras:
        a2 = argparse.Namespace(**vars(args)); a2.steps = max(3, min(args.steps, 8))
        try:
            r64 = measure_batch(a2, prec, rank, world, local, 64, full=False)
            workloads["batch64_1gpu"] = {"workload": "64 x 10 s per GPU (configs[3]'s per-GPU share) on ONE GPU: the weak-scaling base of the N > 1 lines",
                                         "value": r64["value"], "ms_per_step": r64["ms_per_step"], "e2e": r64["e2e"]["value"]}
            del r64
        except Exception as e:
            workloads["batch64_1gpu"] = {"error": f"{type(e).__name__}: {e}"}
        gc.collect(); torch.cuda.empty_cache()
        for other in [m for m in ("fp16", "bf16", "tf32") if m != prec][:2]:
            try:
                r2 = measure_batch(a2, other, rank, world, local, B, full=False)
                rep2 = r2["rep"]
                modes[other] = {"dtype": DTYPE[other], "value": r2["value"], "ms_per_step": r2["ms_per_step"], "e2e": r2["e2e"]["value"],
                                "roofline": roofline_from(rep2, B, L_by_stack, other, peaks, peaks_src, sum(r["ms"] for r in rep2.values())),
                                "breakdown_ms": r2["breakdown_ms"],
                                "parity": parity_of(r2["eng"], run.wav, run.out, other) if run is not None else None}
                del r2
            except Exception as e:
                modes[other] = {"error": f"{type(e).__name__}: {e}"}
            gc.collect(); torch.cuda.empty_cache()
        try:
            workloads["cli_folder"] = wl_cli(prec)
        except Exception as e:
            workloads["cli_folder"] = {"error": f"{type(e).__name__}: {e}"}
        gc.collect(); torch.cuda.empty_cache()
        try:
            lib_base = torch_gpu_result(args, B)
        except Exception as e:
            lib_base = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPE[prec], "data": "synthetic",
            "config": {"workload": (f"configs[2]: batch {B} x {args.seconds:g} s synthetic degraded 44.1 kHz mono utterances, mode 0, "
                                    "seeded synthetic checkpoints, 1 GPU") if world == 1 else
                                   (f"configs[3]: {world * B} x {args.seconds:g} s utterances batch-sharded over {world} GPUs "
                                    f"({B} per GPU), mode 0, NCCL weight broadcast + waveform gather"),
                       "precision": prec, "global_batch": world * B,
                       "launch": "CUDA graph replay of the step's launch sequence" if res["graph"] else "individual launches",
                       "l2": f"no flush needed: {res['ws_gb']:.1f} GB of activations per step >> 126 MB L2",
                       "parallelism": f"batch-shard x{world}: 2 collectives -- NCCL weight broadcast {res['bcast_ms']:.1f} ms (once, start-up) "
                                      "and one waveform gather per step on a side stream" if world > 1 else "single GPU"},
            "e2e": res["e2e"], "gpu_launches": res["gpu_launches"], "clocks": res["clocks"], "roofline": roofline,
            "cpu_baseline": cpu_baseline, "parity": parity, "modes": modes, "workloads": workloads,
            "gpu_library_baseline": lib_base, "breakdown_ms": res["breakdown_ms"],
        }))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    bad = [m for m, p in ([(prec, parity)] + [(k, v.get("parity")) for k, v in modes.items() if isinstance(v, dict)]) if p and not p["ok"]]
    if bad:
        print(f"[bench] PARITY OUT OF TOLERANCE for {bad}: the measurement above is not valid", file=sys.stderr)
        sys.exit(3)


if __name__ == "__main__":
    main()
