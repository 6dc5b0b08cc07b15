#!/usr/bin/env python
"""Benchmark of the vietTTS hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2], the one the metric is quoted on): per GPU a batch of 32
synthetic 100-phoneme / 5 s utterances (N = 312 mel frames, 79 872 samples each) goes through
the NAT acoustic model (encoder, Gaussian upsampling, autoregressive decoder with prenet
dropout, postnet) and the HiFiGAN generator.  One "step" = one such batch.  Weak scaling: every
rank gets its own 32 utterances; the weights are broadcast once from rank 0 over NCCL.

  value  : audio samples / s, whole job, inputs resident in HBM (device-pointer C ABI), CUDA events
  e2e    : same metric through the host-buffer C ABI call (vtts_synthesize_host) with numpy inputs:
           H2D of tokens/durations and D2H of the waveform inside the timed region
  roofline: HiFiGAN generator (98 % of the FLOPs): algorithmic 614.1 MFLOP per mel frame / measured
           stage time (CUDA events recorded around the stage inside the timed region)
  cpu_baseline: the oracle port (torch CPU restatement of the reference) on the host cores,
           bounded sample of the same workload.
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

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

from viettts_b200 import config as C  # noqa: E402
from viettts_b200 import synthetic  # noqa: E402

METRIC = "audio_samples_per_sec"
UNIT = "samples/s"


def peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm_gbs=d.get("hbm_gbs", 6650.0), bf16_tflops=d.get("bf16_tflops", 1590.0),
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", 1400.0), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, budget=DUMP_BUDGET_BYTES):
    """Writes each array as <out_dir>/<name>.npy in float32.  If together they exceed `budget` bytes, every array is
    replaced by a flat sample of its elements (sorted indices drawn with a fixed seed from the array's size) of a size
    proportional to its share, so that two builds run with the same arguments store the same positions."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    room = budget - 1024 * len(arrays)          # leaves room for the .npy headers
    for name, a in arrays.items():
        if total > room:
            k = max(1, room * a.size // total)
            idx = np.sort(np.random.default_rng(a.size).choice(a.size, size=k, replace=False))
            a = a.reshape(-1)[idx]
        np.save(out_dir / f"{name}.npy", a)


def make_batch(batch: int, phonemes: int, seconds: float, seed0: int):
    toks, durs, nfs = [], [], []
    for b in range(batch):
        tk, d = synthetic.utterance(seed0 + b, phonemes, seconds)
        d = (np.asarray(d, np.float32) * np.float32(C.SAMPLE_RATE)) / np.float32(C.HOP)
        toks.append(np.asarray(tk, np.int32))
        durs.append(d[0])
        nfs.append(int(np.sum(d, dtype=np.float32)))
    return np.stack(toks), np.stack(durs).astype(np.float32), np.asarray(nfs, np.int32)


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampler running beside the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------------
# CPU legs (oracle port) -- the only place bench.py executes oracle/
# ---------------------------------------------------------------------------------------------
_CPU_THREADS = None


def cpu_pick_threads(hp, ck):
    """The oracle port is a torch CPU program: the autoregressive part is a Python loop over small
    matmuls (best with few threads), the generator is conv-bound (best with many).  Pick, per stage,
    the fastest thread count on a tiny probe so that the CPU arm is not handicapped by
    oversubscription on a 100+-thread host."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        return _CPU_THREADS
    import torch
    from oracle import hifigan_oracle, nat_oracle
    cores = os.cpu_count() or 1
    tokens, durs, nfs = make_batch(1, 20, 0.4, 7)
    mel = synthetic.mel_input(1, 1, 96)               # long enough that the conv threading of a 5 s utterance shows

    def t_nat():
        with torch.no_grad():
            nat_oracle.inference(ck, tokens, durs, int(nfs[0]), None)

    def t_hg():
        with torch.no_grad():
            hifigan_oracle.generator_forward(hp, mel)

    best = {}
    for name, fn, cands in (("nat", t_nat, [1, 2, 4, 8, 16]), ("hifigan", t_hg, [8, 16, 32, 64, cores])):
        res = []
        for n in sorted(set(c for c in cands if c <= cores)):
            torch.set_num_threads(n)
            fn()
            t0 = time.perf_counter()
            fn()
            res.append((time.perf_counter() - t0, n))
        best[name] = min(res)[1]
    _CPU_THREADS = best
    return best


def cpu_port_step(hp, ck, tokens, durs, nfs, masks):
    """One pass of the reference algorithm (torch CPU restatement) over the given utterances, one utterance per call
    like the reference's own predict_mel / mel2wave (a 32-row call is slower per utterance on the host: its
    activations, 135 MB per utterance, fall out of every cache)."""
    import torch
    from oracle import hifigan_oracle, nat_oracle
    th = cpu_pick_threads(hp, ck)
    total = 0
    with torch.no_grad():
        for r in range(tokens.shape[0]):
            torch.set_num_threads(th["nat"])
            mel = nat_oracle.inference(ck, tokens[r:r + 1], durs[r:r + 1], int(nfs[r]), masks[r:r + 1])
            torch.set_num_threads(th["hifigan"])
            wav = hifigan_oracle.generator_forward(hp, mel.numpy())
            total += int(wav.numel())
    return total


def cpu_baseline(hp, ck, phonemes, seconds, budget_s=12.0, rows=1):
    th = cpu_pick_threads(hp, ck)
    tokens, durs, nfs = make_batch(rows, phonemes, seconds, 9000)
    masks = synthetic.dropout_masks(3, rows, int(nfs[0]))
    cpu_port_step(hp, ck, tokens[:1], durs[:1], nfs[:1], masks[:1])  # warm-up
    t0 = time.perf_counter()
    samples, it = 0, 0
    while True:
        samples += cpu_port_step(hp, ck, tokens, durs, nfs, masks)
        it += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return dict(value=samples / dt, unit=UNIT, cores=max(th.values()), kind="port",
                sample=f"{it} passes of {rows} utterance(s) ({phonemes} phonemes, {int(nfs[0])} frames) through oracle/ (torch CPU; "
                       f"threads: acoustic {th['nat']}, generator {th['hifigan']} of {os.cpu_count()} host threads, picked by a probe), {dt:.1f} s")


def run_reference(args):
    """--impl reference: the reference algorithm's CPU implementation (oracle port; the
    reference's JAX/Haiku path cannot be installed offline), best host thread counts."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    hp = synthetic.hifigan_params(1234)
    ck = synthetic.acoustic_ckpt(1234)
    th = cpu_pick_threads(hp, ck)
    rows = args.ref_rows
    tokens, durs, nfs = make_batch(rows, args.phonemes, args.seconds, 0)
    masks = synthetic.dropout_masks(3, rows, int(nfs[0]))
    t0 = time.perf_counter()
    cpu_port_step(hp, ck, tokens[:1], durs[:1], nfs[:1], masks[:1])      # one warm-up pass (the CPU port has no compile / cache state to warm)
    t_row = time.perf_counter() - t0
    # bounded sample: keep the whole run near the budget (default 150 s) by trimming the rows of a step, never below one
    cap = max(1, int(args.ref_budget_s / max(args.steps, 1) / max(t_row, 1e-3)))
    if cap < rows:
        rows = cap
        tokens, durs, nfs, masks = tokens[:rows], durs[:rows], nfs[:rows], masks[:rows]
    t0 = time.perf_counter()
    samples = 0
    for _ in range(args.steps):
        samples += cpu_port_step(hp, ck, tokens, durs, nfs, masks)
    dt = time.perf_counter() - t0
    val = samples / dt
    desc = (f"{args.steps} steps x {rows} utterance(s) of the batch-{args.batch} workload, one utterance per call, through oracle/ (torch CPU "
            f"restatement; threads: acoustic {th['nat']}, generator {th['hifigan']} of {os.cpu_count()} host threads)")
    out = dict(metric=METRIC, value=val, unit=UNIT, impl="reference", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
               ms_per_step=1e3 * dt / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
               rtf=(dt / (samples / C.SAMPLE_RATE)),
               config=workload_config(args, int(os.environ.get("WORLD_SIZE", "1"))),
               cpu_baseline=dict(value=val, unit=UNIT, cores=max(th.values()), kind="port", sample=desc),
               e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
# algorithmic FLOPs per mel frame of each generator sub-stage (SURVEY.md §8a/§8d: 2 x MACs; sums to 614 105 088)
_HG_MAC = dict(conv_pre=7 * 80 * 512, conv_post=256 * 7 * 32,
               stage0=8 * 256 * 256 * 126 + 8 * 2 * 512 * 256, stage1=64 * 128 * 128 * 126 + 64 * 2 * 256 * 128,
               stage2=128 * 64 * 64 * 126 + 128 * 2 * 128 * 64, stage3=256 * 32 * 32 * 126 + 256 * 2 * 64 * 32)
assert 2 * sum(_HG_MAC.values()) == C.HIFIGAN_FLOP_PER_FRAME, sum(_HG_MAC.values())


def workload_config(args, world):
    """The `config` object both arms print (identical content, so the driver's same_config check can hold)."""
    n = int(args.seconds * C.SAMPLE_RATE / C.HOP)
    return dict(workload=f"NAT acoustic + HiFiGAN, {args.phonemes}-phoneme / {args.seconds:g} s utterances, batch {args.batch} per GPU (BASELINE configs[2])",
                batch_per_gpu=args.batch, phonemes=args.phonemes, mel_frames=n, samples_per_utterance=n * C.HOP,
                parallelism=f"utterance-sharded x{world}",
                l2="activations per step (>4 GB) exceed the 126 MB L2; no flush needed", dropout="on-device threefry keep-masks")


class Job:
    """One batch resident on the device + the calls that time it."""

    def __init__(self, eng, dev, tokens, durs, nfs, seed, lengths=None):
        import torch
        self.eng, self.dev = eng, dev
        self.tokens, self.durs, self.nfs, self.seed, self.lengths = tokens, durs, nfs, seed, lengths
        self.B, self.L = tokens.shape
        self.N = int(nfs.max())
        self.tok_t = torch.from_numpy(tokens).to(dev)
        self.dur_t = torch.from_numpy(durs).to(dev)
        self.nf_t = torch.from_numpy(nfs).to(dev)
        self.len_t = None if lengths is None else torch.from_numpy(lengths).to(dev)
        self.mel_t = torch.empty((self.B, self.N, C.MEL_DIM), dtype=torch.float32, device=dev)
        self.wav_t = torch.empty((self.B, self.N * C.HOP), dtype=torch.float32, device=dev)
        self.samples = int(nfs.sum()) * C.HOP
        self.frames = int(nfs.sum())

    def step(self, marks=None):
        e = self.eng
        if marks is not None:
            marks[0].record()
        e.acoustic_forward(self.tok_t, self.dur_t, self.N, lengths_t=self.len_t, n_frames_t=self.nf_t, seed=self.seed, out=self.mel_t)
        if marks is not None:
            marks[1].record()
        e.hifigan_forward(self.mel_t, self.nf_t, out=self.wav_t)
        if marks is not None:
            marks[2].record()


def time_jobs(jobs, steps, warmup, barrier):
    """CUDA-event time of `steps` passes over the jobs of this rank (device-resident inputs)."""
    import torch
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    for _ in range(warmup):
        for j in jobs:
            j.step()
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    marks = [[[ev(), ev(), ev()] for _ in jobs] for _ in range(steps)]
    e0, e1 = ev(), ev()
    e0.record()
    for k in range(steps):
        for ji, j in enumerate(jobs):
            j.step(marks[k][ji])
    e1.record()
    torch.cuda.synchronize()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    ac = float(np.sum([[m[0].elapsed_time(m[1]) for m in row] for row in marks])) / steps
    hg = float(np.sum([[m[1].elapsed_time(m[2]) for m in row] for row in marks])) / steps
    return ms, ac, hg


def time_e2e(eng, job, steps, out):
    """Wall time of `steps` host-buffer calls (numpy in -> H2D -> kernels -> D2H -> numpy out)."""
    for _ in range(2):
        eng.synthesize(job.tokens, job.durs, lengths=job.lengths, n_frames=job.nfs, seed=job.seed, out=out)
    t0 = time.perf_counter()
    for _ in range(steps):
        w = eng.synthesize(job.tokens, job.durs, lengths=job.lengths, n_frames=job.nfs, seed=job.seed, out=out)
    return (time.perf_counter() - t0) / steps, w


def stage_rooflines(eng, job, pk, precision):
    """One entry per kernel group of the step: device ms (CUDA events between the kernels, vtts_debug_substages), the
    algorithmic work of SURVEY.md §8(d) and the bound it is measured against."""
    import torch
    eng.substages(True)
    job.step()
    torch.cuda.synchronize()
    ms = eng.substages(False)
    rows, frames = job.B, job.frames
    hbm = pk["hbm_gbs"]
    tc_ceiling = pk["bf16_tflops_sustained"] / 3.0 if precision != "fp32" else 74.4
    out = {}

    def tensor(name, key, flop, note=None):
        if key not in ms:
            return
        t = flop / (ms[key] / 1e3) / 1e12
        out[name] = dict(ms=ms[key], bound="tensor (bf16x3: 1/3 of the measured sustained bf16 peak)" if precision != "fp32" else "fp32 FMA pipe",
                         achieved_tflops=t, frac_of_ceiling=t / tc_ceiling, algorithmic_flop=flop)
        if note:
            out[name]["note"] = note

    for i in range(4):
        tensor(f"hifigan_stage{i}", f"hifigan.stage{i}", 2.0 * _HG_MAC[f"stage{i}"] * frames)
    tensor("hifigan_conv_pre", "hifigan.conv_pre", 2.0 * _HG_MAC["conv_pre"] * frames)
    if "hifigan.conv_post" in ms:
        byts = frames * 256 * (3 * 32 * 4 + 4)          # reads the three ResBlock outputs, writes one sample
        g = byts / (ms["hifigan.conv_post"] / 1e3) / 1e9
        out["hifigan_conv_post"] = dict(ms=ms["hifigan.conv_post"], bound="hbm", achieved_gbs=g, frac_hbm=g / hbm, algorithmic_bytes=byts)
    if "acoustic.decoder_scan" in ms:
        t = ms["acoustic.decoder_scan"]
        launches = (rows + 127) // 128
        out["nat_decoder_scan"] = dict(ms=t, bound="latency (sequential over frames; weights resident on chip)", us_per_frame=1e3 * t / (job.N * launches),
                                       rows=rows, frames=job.N, achieved_tflops_fp32=12_918_784.0 * frames / (t / 1e3) / 1e12,
                                       note="12 918 784 FLOP per frame per row (SURVEY 8d); cond projections hoisted into acoustic.cond_gemm")
    tensor("nat_cond_gemm", "acoustic.cond_gemm", 2.0 * 512 * 4096 * frames, "hoisted cond . W[0:512] of both decoder LSTMs")
    tensor("nat_postnet", "acoustic.postnet", 8_683_520.0 * frames)
    tensor("nat_projection", "acoustic.projection", 2.0 * 1024 * 80 * frames)
    if "acoustic.upsample" in ms:
        byts = rows * job.L * 2048 + frames * 2048
        g = byts / (ms["acoustic.upsample"] / 1e3) / 1e9
        out["nat_upsample"] = dict(ms=ms["acoustic.upsample"], bound="hbm/L2", achieved_gbs=g, frac_hbm=g / hbm, algorithmic_bytes=byts)
    if "acoustic.encoder" in ms:
        out["nat_token_encoder"] = dict(ms=ms["acoustic.encoder"], bound="latency (BiLSTM scan over tokens)", us_per_token=1e3 * ms["acoustic.encoder"] / job.L)
    return out


def c5_workload(n=256, seed0=5000):
    """BASELINE configs[4]: n utterances, L ~ U{50..300} phonemes at ~0.05 s per phoneme."""
    rng = np.random.default_rng(77)
    utts = []
    for i in range(n):
        L = int(rng.integers(50, 301))
        tk, d = synthetic.utterance(seed0 + i, L, None)
        d = (np.asarray(d, np.float32) * np.float32(C.SAMPLE_RATE)) / np.float32(C.HOP)
        utts.append((np.asarray(tk, np.int32), d[0], int(np.sum(d, dtype=np.float32))))
    return utts


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from viettts_b200 import parallel
    from viettts_b200.engine import Engine

    eng = Engine(local)
    eng.set_precision(args.precision)
    if args.tc_variant is not None:
        eng.tc_stats(False, variant=args.tc_variant)
    if args.pairs != "auto":
        eng.set_fused_pairs(args.pairs != "off", kind=None if args.pairs == "off" else args.pairs)
    hp = synthetic.hifigan_params(1234) if rank == 0 else None
    ck = synthetic.acoustic_ckpt(1234) if rank == 0 else None
    t_w = time.perf_counter()
    wbytes = parallel.load_weights_distributed(eng, hp, ck, dev)
    t_w = time.perf_counter() - t_w

    def barrier():
        if world > 1:
            dist.barrier()

    def allmax(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allgather(x):
        if world == 1:
            return [float(x)]
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        outl = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(outl, t)
        return [float(o.item()) for o in outl]

    W = max(args.warmup, 3)
    side_steps = max(3, min(args.steps, 5))
    pk = peaks()

    # ================= headline: BASELINE configs[2], weak scaling, 32 utterances per GPU =================
    B = args.batch
    tokens, durs, nfs = make_batch(B, args.phonemes, args.seconds, 1000 * rank)
    job = Job(eng, dev, tokens, durs, nfs, 0xC0FFEE + rank)
    N, L = job.N, job.L
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count()
    ms_step, ac_ms, hg_ms = time_jobs([job], args.steps, W, barrier)
    # the last timed step's results, taken before the lines below run other work through the same buffers
    dumped = dict(mel=job.mel_t.cpu().numpy(), wav=job.wav_t.cpu().numpy()) if args.dump_outputs and rank == 0 else None
    launches = (eng.launch_count() - l0) * args.steps // (args.steps + W)
    clocks = sampler.stop() if rank == 0 else None
    ms_step = allmax(ms_step)
    value = world * job.samples / (ms_step / 1e3)

    # ---- e2e through the host-buffer C ABI: page-locked result buffer (headline) and a pageable numpy result ----
    wav_pinned = Engine.pinned_empty((B, N * C.HOP))
    barrier()
    dt, wav_h = time_e2e(eng, job, args.steps, wav_pinned)
    dt = allmax(dt)
    e2e_val = world * job.samples / dt
    dt_pg, _ = time_e2e(eng, job, side_steps, np.empty((B, N * C.HOP), np.float32))
    dt_pg = allmax(dt_pg)
    h2d = tokens.nbytes + durs.nbytes + nfs.nbytes
    d2h = wav_h.nbytes

    def line_for(jobs, steps, scaling_world=world, e2e_job=None):
        ms, ac, hg = time_jobs(jobs, steps, 3, barrier)
        per_rank = allgather(ms)
        ms_max = max(per_rank)
        samples = sum(j.samples for j in jobs)
        tot = samples
        if world > 1:
            t = torch.tensor([samples], dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            tot = float(t.item())
        d = dict(value=tot / (ms_max / 1e3), unit=UNIT, ms_per_step=ms_max, stages_ms=dict(acoustic=ac, hifigan=hg),
                 rtf=(ms_max / 1e3) / (tot / C.SAMPLE_RATE), per_rank_busy_ms=per_rank,
                 imbalance_max_over_mean=ms_max / (sum(per_rank) / len(per_rank)))
        if e2e_job is not None:
            o = Engine.pinned_empty((e2e_job.B, e2e_job.N * C.HOP))
            dte, _ = time_e2e(eng, e2e_job, steps, o)
            d["e2e_value"] = e2e_job.samples / dte
        return d

    # ================= batch sweep and strict-fp32 line (N = 1 only; north_star: batch 1/8/32/128) =================
    sweep, strict = None, None
    if world == 1 and not args.no_sweep:
        sweep = {str(B): dict(value=value, ms_per_step=ms_step, stages_ms=dict(acoustic=ac_ms, hifigan=hg_ms), e2e_value=e2e_val,
                              rtf=(ms_step / 1e3) / (job.samples / C.SAMPLE_RATE))}
        for b2 in (1, 8, 128):
            if b2 == B:
                continue
            t2, d2, n2 = make_batch(b2, args.phonemes, args.seconds, 7000)
            j2 = Job(eng, dev, t2, d2, n2, 0xC0FFEE)
            r = line_for([j2], side_steps, e2e_job=j2)
            sweep[str(b2)] = {k: r[k] for k in ("value", "ms_per_step", "stages_ms", "e2e_value", "rtf")}
            del j2
        if args.precision != "fp32":
            eng.set_precision("fp32")
            r = line_for([job], 3, e2e_job=job)
            strict = dict(dtype="f32 (IEEE fp32 FMA on the CUDA cores, conv1d.cu)", batch=B,
                          **{k: r[k] for k in ("value", "ms_per_step", "stages_ms", "e2e_value", "rtf")})
            eng.set_precision(args.precision)

    # ================= BASELINE configs[3]: 128 utterances sharded over the ranks (strong scaling) =================
    configs = {}
    if not args.no_configs:
        tk4, du4, nf4 = make_batch(128, args.phonemes, args.seconds, 31000)
        shard = sorted(parallel.lpt_shard(nf4, world)[rank])
        j4 = Job(eng, dev, tk4[shard], du4[shard], nf4[shard], 0xC4)
        r = line_for([j4], side_steps)
        configs["c4"] = dict(workload="128 x 100-phoneme / 5 s utterances, LPT-sharded by n_frames over the ranks (BASELINE configs[3])",
                             scaling="strong", rows_per_gpu=len(shard), **r)
        del j4
        # ================= BASELINE configs[4]: n=256 mixed 50-300 phonemes, bucketed <= 8 % padding =================
        utts = c5_workload()
        nfs5 = [u[2] for u in utts]
        # equal-cost contiguous buckets (a multiple of the rank count), LPT-assigned: parallel.balanced_buckets
        buckets, shards5 = parallel.balanced_buckets(nfs5, world, groups_per_rank=args.c5_groups or None, max_pad_frac=0.08, max_rows=32)
        mine = shards5[rank]
        jobs5 = []
        for bi in mine:
            bk = buckets[bi]
            Lm = max(len(utts[i][0]) for i in bk)
            tk = np.zeros((len(bk), Lm), np.int32)
            du = np.zeros((len(bk), Lm), np.float32)
            ln = np.zeros(len(bk), np.int32)
            for r_, i in enumerate(bk):
                tk[r_, : len(utts[i][0])] = utts[i][0]
                du[r_, : len(utts[i][0])] = utts[i][1]
                ln[r_] = len(utts[i][0])
            jobs5.append(Job(eng, dev, tk, du, np.asarray([nfs5[i] for i in bk], np.int32), 0xC5, lengths=ln))
        r = line_for(jobs5, side_steps)
        padded = sum(len(bk) * max(nfs5[i] for i in bk) for bk in buckets)
        configs["c5"] = dict(workload="256 utterances, 50-300 phonemes (156-937 frames), bucketed by frame count and LPT-assigned to the ranks "
                                      "(BASELINE configs[4])", scaling="strong", n_utterances=len(utts), n_buckets=len(buckets),
                             buckets_per_rank=len(buckets) / world, rows_per_bucket=[len(bk) for bk in buckets], padding_frac=1.0 - sum(nfs5) / padded, buckets_on_this_rank=len(mine), **r)
        del jobs5

    # ================= per-stage rooflines (rank 0) =================
    stages = stage_rooflines(eng, job, pk, args.precision) if rank == 0 else None

    # ---- STFT/log-mel kernel (MelFilter, nat/dsp.py:104-128), measured separately ----
    mel_info = None
    if rank == 0:
        ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
        S = 79872
        MB = 512                                     # 512 x 5 s = 164 MB of samples: larger than L2
        wav_m = torch.rand((MB, S), dtype=torch.float32, device=dev) - 0.5
        mel_m = torch.empty((MB, S // C.HOP, C.MEL_DIM), dtype=torch.float32, device=dev)
        for _ in range(3):
            eng.melspec_forward(wav_m, out=mel_m)
        m0, m1 = ev(), ev()
        m0.record()
        for _ in range(5):
            eng.melspec_forward(wav_m, out=mel_m)
        m1.record()
        torch.cuda.synchronize()
        mms = m0.elapsed_time(m1) / 5
        mbytes = MB * S * 5.25                      # 4 B in + 1.25 B out per sample (SURVEY 8d)
        mflop = MB * (S // C.HOP) * 29704.0         # sparse-filterbank FLOP count per frame (SURVEY 8d)
        mel_info = dict(samples_per_s=MB * S / (mms / 1e3), ms=mms, achieved_gbs=mbytes / (mms / 1e3) / 1e9,
                        peak_gbs=pk["hbm_gbs"], frac_hbm=mbytes / (mms / 1e3) / 1e9 / pk["hbm_gbs"],
                        achieved_tflops_fp32=mflop / (mms / 1e3) / 1e12, batch=MB, samples_per_row=S,
                        fp32_peak_tflops=74.4, frac_fp32=mflop / (mms / 1e3) / 1e12 / 74.4,
                        note="one warp per frame pair, FFT-1024 = 32 x 32 four-step with register-resident 32-point transforms; arithmetic intensity "
                             "22 FLOP/B sits above the FP32 ridge (11 FLOP/B): the kernel is FP32-issue bound, not HBM bound")
        if stages is not None:
            stages["melspec"] = dict(ms=mms, bound="hbm target (SURVEY 8d), fp32-issue bound in practice", achieved_gbs=mel_info["achieved_gbs"],
                                     frac_hbm=mel_info["frac_hbm"], frac_fp32=mel_info["frac_fp32"])
        del wav_m, mel_m

    # ---- callers of the path (SURVEY 8f): duration model + one-call token->wav, chunked vocoding latency, GTA ----
    callers = None
    if rank == 0 and world == 1 and not args.no_callers:
        seed = job.seed
        eng.load_duration(synthetic.duration_ckpt(1234))
        for _ in range(2):
            waves, _ = eng.tts(tokens, silence_duration=0.05, seed=seed)
        t0 = time.perf_counter()
        reps = max(3, min(args.steps, 10))
        for _ in range(reps):
            waves, _ = eng.tts(tokens, silence_duration=0.05, seed=seed)
        dt_tts = (time.perf_counter() - t0) / reps
        tts_samples = int(sum(w.size for w in waves))
        dur_ms = eng.last_stage_ms(3)
        mel1 = synthetic.mel_input(3, 1, N)
        for _ in range(2):
            next(eng.mel2wave_stream(mel1, chunk_frames=32))
        t0 = time.perf_counter()
        for _ in range(10):
            next(eng.mel2wave_stream(mel1, chunk_frames=32))
        first_ms = (time.perf_counter() - t0) / 10 * 1e3
        t0 = time.perf_counter()
        n_stream = sum(p.size for p in eng.mel2wave_stream(mel1, chunk_frames=32))
        all_ms = (time.perf_counter() - t0) * 1e3
        eng.load_mel_filterbank()
        S_g = N * C.HOP
        wav_i16 = (np.random.default_rng(1).standard_normal((B, S_g)) * 3000).astype(np.int16)
        dur_sec = durs * np.float32(C.HOP / C.SAMPLE_RATE)
        for _ in range(2):
            eng.gta(wav_i16, tokens, dur_sec, seed=seed)
        eng.substages(True)
        t0 = time.perf_counter()
        for _ in range(reps):
            eng.gta(wav_i16, tokens, dur_sec, seed=seed)
        dt_gta = (time.perf_counter() - t0) / reps
        gta_dev_ms = eng.last_stage_ms(1)
        gta_sub = {k: v for k, v in eng.substages(False).items() if k.startswith("teacher.")}
        callers = dict(
            gta=dict(api="vtts_gta_host (int16 audio -> log-mel -> shift -> teacher-forced acoustic model, zoneout + dropout on), host buffers",
                     batch=B, frames_per_s=B * N / dt_gta, ms_per_call=dt_gta * 1e3, teacher_forced_model_ms=gta_dev_ms,
                     teacher_forced_stages_ms=gta_sub, autoregressive_model_ms=ac_ms),
            text_to_wav=dict(api="vtts_tts_host (duration model -> duration fix-ups -> acoustic -> trailing-silence trim -> generator), host buffers",
                             batch=B, samples_per_s=tts_samples / dt_tts, ms_per_call=dt_tts * 1e3, samples_per_call=tts_samples,
                             duration_model_ms=dur_ms),
            streaming_vocoder=dict(api="Engine.mel2wave_stream, B=1, 32-frame chunks + 16-frame recomputed halo, host buffers",
                                   first_chunk_ms=first_ms, audio_ms_per_chunk=32 * C.HOP / C.SAMPLE_RATE * 1e3,
                                   whole_utterance_ms=all_ms, samples=n_stream))

    if rank == 0:
        frames = job.frames
        flops = frames * C.HIFIGAN_FLOP_PER_FRAME
        ach = flops / (hg_ms / 1e3) / 1e12
        traffic, traffic_src = None, None
        for tp in sorted((REPO / "profiles").glob("r*_traffic.json"), reverse=True):
            tj = json.loads(tp.read_text())
            w = tj.get("workload", {})
            if w.get("batch") == B and w.get("mel_frames") == N and w.get("precision") == args.precision and w.get("pairs", "auto") == args.pairs:
                traffic = tj["generator_dram_bytes_per_step"]
                traffic_src = f"sum of dram__bytes_read+write over the generator launches of one step, ncu launch list of this command ({tp.name}); not re-measured in this run"
                break
        ceiling = pk["bf16_tflops_sustained"] / 3.0 if args.precision != "fp32" else 74.4
        out = dict(
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=W, ms_per_step=ms_step,
            higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype="f32" if args.precision == "fp32" else "f32 (bf16x3 split products on tcgen05, fp32 accumulate/storage)", data="synthetic",
            rtf=(ms_step / 1e3) / (world * job.samples / C.SAMPLE_RATE),
            config=workload_config(args, world),
            stages_ms=dict(acoustic=ac_ms, hifigan=hg_ms),
            e2e=dict(value=e2e_val, unit=UNIT, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h), ms_per_step=1e3 * dt,
                     api="vtts_synthesize_host via viettts_b200.Engine.synthesize (numpy in; numpy out in a page-locked buffer the D2H copy lands in)",
                     pageable_result=dict(value=world * job.samples / dt_pg, ms_per_step=1e3 * dt_pg,
                                          note="same call with a plain numpy result array (the reference's return type): one more host copy")),
            gpu_launches=int(launches),
            roofline=dict(bound="tensor",
                          kernel=("tcgen05 conv kernels of the generator (tc_conv_kernel, CTA-pair form for C >= 128, + tc_pair2_kernel), all launches of one step (+ conv_post, 1 % of the stage time)"
                                  if args.precision != "fp32" else "conv1d_nwc_kernel: the generator launches of one step (+ conv_post)"),
                          achieved=ach, peak=pk["bf16_tflops_sustained"], unit="TFLOP/s", frac=ach / pk["bf16_tflops_sustained"],
                          traffic=traffic, traffic_source=traffic_src,
                          algorithmic_flops_per_step=flops, launch_ms=hg_ms,
                          frac_of_mode_ceiling=ach / ceiling,
                          mode_ceiling=("1/3 of the bf16 peak: bf16x3 issues three bf16 MMAs per algorithmic product" if args.precision != "fp32"
                                        else "FP32 FMA pipe, nominal 74.4 TFLOP/s"),
                          peak_source=pk["source"] + ", sustained bf16 dense",
                          note=("algorithmic fp32 FLOPs; the bf16x3 path issues 3 bf16 MMAs per algorithmic product, so 1/3 of the bf16 peak is its ceiling"
                                if args.precision != "fp32" else "strict-fp32 path runs on the FP32 FMA pipe (nominal 74 TFLOP/s)")),
            roofline_stages=stages,
            clocks=clocks, weights=dict(bytes=wbytes, broadcast_s=t_w), melspec=mel_info, callers=callers,
            sweep=sweep, strict_fp32=strict, configs=configs or None,
        )
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline(synthetic.hifigan_params(1234), synthetic.acoustic_ckpt(1234), args.phonemes, args.seconds)
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(out))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--phonemes", type=int, default=100)
    ap.add_argument("--seconds", type=float, default=5.0)
    ap.add_argument("--ref-rows", type=int, default=32, help="utterances per step of the CPU reference arm (default: the GPU arm's batch)")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="wall-time target of the whole reference-arm run; a step is trimmed to fewer rows if needed")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-callers", action="store_true", help="skip the duration/tts/gta/streaming side measurements (profiling runs)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the batch sweep and the strict-fp32 line")
    ap.add_argument("--no-configs", action="store_true", help="skip BASELINE configs[3] / configs[4]")
    ap.add_argument("--c5-groups", type=int, default=0, help="equal-cost buckets per rank of the mixed-length workload (0 = pick 2..4 by predicted makespan)")
    ap.add_argument("--pairs", default="auto", choices=["auto", "off", "smem2", "smem2c", "tmem", "smem"],
                    help="C<=64 ResBlock pairs: auto = library default, off = two conv launches per pair, tmem / smem = fused pair kernel "
                         "with the A operand in tensor memory / shared memory")
    ap.add_argument("--tc-variant", type=int, default=None, help="tile-shape variant of tc_conv (tuning aid; default: library default)")
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "fp32"],
                    help="conv arithmetic: bf16x3 = tcgen05 split-bf16 with fp32 accumulate (default), fp32 = FMA pipe")
    ap.add_argument("--dump-outputs", type=Path, default=None, metavar="DIR",
                    help="after the timed steps write what the last one computed for rank 0's batch, mel [B,N,80] and wav [B,256N], "
                         "as DIR/mel.npy and DIR/wav.npy (float32, at most 64 MB in all: a fixed, seeded sample beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
