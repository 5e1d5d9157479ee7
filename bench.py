#!/usr/bin/env python
"""bench.py — RTF / mel-frames-per-second of the F5-TTS ODE-sampling hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2|cfg3|cfg4|cfg5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of synthetic utterances:
    mel front-end (STFT kernel) -> CFM.sample (NFE x backbone + CFG + Euler) -> Vocos decode (ISTFT kernel).
Headline workload = BASELINE.json configs[1] ("cfg2"): F5-TTS Base, batch 1, 10 s total (938 frames, 282 prompt frames),
NFE 32, cfg 2.0, sway -1.0, random-init weights in the released checkpoint layout (SURVEY.md §8d), fp16 tensor-core
operands with fp32 accumulation / residual / ODE state.  With --gpus N every rank runs the same workload on its own
GPU (weak scaling, utterances are independent) and all-gathers the finished mel + audio each step (NCCL).

Keys of the JSON line:
`value`     generated mel frames per second, whole job, inputs already resident in HBM.
`e2e`       the same metric through the reference-facing top call `infer_process((audio, sr), ref_text, gen_text, model,
            vocoder, ...)` (utils_infer.py:384-434 mirror) with HOST audio in and a HOST numpy waveform out: H2D, text
            front-end, mel kernel, sampler, vocoder and D2H are all inside the timed region.
`parity`    final-mel rel-L2 of THIS run's sampler against the committed output of the unmodified fp32 reference on the
            same workload and injected y0 (tests/golden/cfg2_full_nfe32.npz), with the drift per step.
`roofline`  every tensor kernel of a block timed alone from a CUDA graph over > L2 of distinct weights; `kernel` is the
            entry with the largest share of the step; `gemm_time_weighted_frac` weights the GEMM fractions by their time;
            `library_ref_us` = the same shape through torch.matmul (cuBLAS) / F.scaled_dot_product_attention, the
            kernels the reference would dispatch to on this GPU (SURVEY.md §2.1) — comparators, never on the hot path;
            `step_tensor` = whole-step algorithmic FLOP/s against the sustained peak; `bandwidth_kernels` = achieved
            GB/s of the HBM/L2-bound kernels against the measured copy bandwidth.
`workloads` further BASELINE.json configurations measured in the same run: cfg3 (batch 8, variable length) and cfg5
            (E2-TTS) on one GPU, and cfg4 = 64 utterances x NFE 16 sharded over all N ranks (`plan_shards`, batches of 8,
            one padded NCCL all-gather of mel + audio at the end; strong scaling: the global batch is fixed).
`cpu_baseline` / --impl reference  the CPU oracle port of the reference (oracle/f5_oracle.py, fp32, all granted host
            cores); see `reference_arm`.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import synthdata as SD  # noqa: E402  (neutral synthetic weights / inputs shared with the tests and the CPU oracle)

WORKLOADS = SD.WORKLOADS
CFG_STRENGTH, SWAY = SD.CFG_STRENGTH, SD.SWAY
synth_inputs = SD.synth_inputs
GOLDEN_CFG2 = os.path.join(ROOT, "tests", "golden", "cfg2_full_nfe32.npz")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d.get("hbm_gbs", 6650.0), tf=d.get("bf16_tflops", 1590.0),
                    tf_sus=d.get("bf16_tflops_sustained", 1400.0), src="MEASURED_PEAKS.json")
    return dict(hbm=6650.0, tf=1590.0, tf_sus=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi sampled every 200 ms DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def __enter__(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = [float(r[1]) for r in rows]
            busy = [v for v in sm if v > 0.5 * max(sm)] or sm
            out["sm_mhz"] = statistics.median(busy)
            out["sm_max_mhz"] = float(rows[0][2])
            out["samples"] = len(rows)
            out["power_w_max"] = max(float(r[3]) for r in rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for i, n in enumerate(names):
                if any("Active" in r[5 + i] and "Not" not in r[5 + i] for r in rows):
                    out["reasons"].append(n)
        except Exception as e:  # noqa: BLE001
            out["error"] = str(e)
        finally:
            if self.path and os.path.exists(self.path):
                os.unlink(self.path)
        return out


_VOCAB = [chr(ord("a") + i) for i in range(26)] + [" ", ".", ","]


def build_gpu_model(arch_name, dev):
    import f5_tts_b200 as F5
    from f5_tts_b200.vocoder import Vocos

    cfg = getattr(SD, arch_name)()
    cls = F5.DiT if cfg.backbone == "DiT" else F5.UNetT
    vocab = {c: i for i, c in enumerate(_VOCAB)}  # only the e2e leg tokenises text; ids stay inside the 2546-row table
    model = F5.CFM(transformer=cls(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, ff_mult=cfg.ff_mult,
                                   text_dim=cfg.text_dim, text_mask_padding=cfg.text_mask_padding,
                                   conv_layers=cfg.conv_layers, pe_attn_head=cfg.pe_attn_head,
                                   text_num_embeds=cfg.text_num_embeds, mel_dim=100), vocab_char_map=vocab)
    model.load_state_dict(SD.synthetic_state_dict(cfg, seed=1234), strict=True)
    voc = Vocos()
    voc.load_state_dict(SD.synthetic_vocos_state_dict(), strict=False)
    return model.to(dev), voc.to(dev), cfg


def hot_path(model, voc, wav, text, duration, lens, nfe, frames0=None, exact_varlen=False):
    """mel front-end + CFM.sample + vocoder; returns (mel [B,N,100], audio [B, nw])."""
    B = wav.shape[0]
    if B == 1:
        out, _ = model.sample(wav, text, frames0 if frames0 is not None else int(duration[0]), steps=nfe,
                              cfg_strength=CFG_STRENGTH, sway_sampling_coef=SWAY, seed=0)
        ref = wav.shape[-1] // 256
    else:
        cond = model.mel_spec(wav, frames_last=False)
        out, _ = model.sample(cond, text, duration, lens=lens, steps=nfe, cfg_strength=CFG_STRENGTH,
                              sway_sampling_coef=SWAY, seed=0, exact_varlen=exact_varlen)
        ref = int(lens.min())
    audio = voc.decode(out[:, ref:, :].permute(0, 2, 1).float())
    return out, audio


def _graph_time_us(fn, n_launch, rounds=5):
    """Average device time per launch of `fn` (which enqueues n_launch kernels): captured into a CUDA graph so that
    host-side launch cost (ctypes + tensor-map encoding) is not in the measurement; CUDA events on the launching stream."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(rounds):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (rounds * n_launch)


def load_traffic():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except Exception:  # noqa: BLE001
        return {}


def isolated_kernel_roofline(cfg, M, seq, peaks, dev):
    """Every tensor kernel of one backbone block timed alone: >= 192 MB of distinct weight matrices (> L2, so every launch
    streams W from HBM as in the real step) launched back to back from a CUDA graph, CUDA events on the launching
    stream.  Beside each: the same contraction through the library kernel the reference dispatches to (cuBLAS via
    torch.matmul fp16 / SDPA), timed the same way — a comparator only."""
    import torch.nn.functional as TF

    from f5_tts_b200 import ops

    g = torch.Generator().manual_seed(3)
    D, F, H = cfg.dim, int(cfg.dim * cfg.ff_mult), cfg.heads
    Be = M // seq
    depth = cfg.depth

    def run(N, K, epi, act, tag, per_step, **kw):
        n_w = max(24, -(-192_000_000 // (N * K * 2)))
        a = [torch.randn(M, K, generator=g).half().to(dev) for _ in range(2)]
        w = [(torch.randn(N, K, generator=g) / 32).half().to(dev) for _ in range(n_w)]
        b = torch.randn(N, generator=g).to(dev)
        if epi == ops.EPI_RESID:
            kw["resid"] = torch.zeros(M, N, device=dev)
            kw["gate"] = torch.randn(N, generator=g).to(dev)
        us = _graph_time_us(lambda: [ops.linear(a[i % 2], w[i], b, epi=epi, act=act, bn=0, pair=0, static_w=True, **kw)
                                     for i in range(n_w)], n_w)
        wt = [x.t() for x in w]  # [K, N] views: torch.matmul(a, w.T) -> cuBLAS NT GEMM, the nn.Linear kernel
        lib = _graph_time_us(lambda: [torch.matmul(a[i % 2], wt[i]) for i in range(n_w)], n_w)
        fl = 2.0 * M * N * K
        tile = ops.gemm_tile(M, N, K, epi, act)
        return dict(kernel=tag, shape=[M, N, K], launches_per_step=per_step,
                    tile=f"{'256' if tile[1] else '128'}x{tile[0]}{' cta_group::2' if tile[1] else ''}",
                    us_per_launch=round(us, 2), tflops=round(fl / us / 1e6, 1), frac=round(fl / us / 1e6 / peaks["tf"], 4),
                    flops_per_launch=fl, library_ref_us=round(lib, 2),
                    library_ref="torch.matmul fp16 (cuBLAS), plain GEMM: no bias / activation / RoPE / residual epilogue")

    rows = [run(F, D, ops.EPI_F16, ops.ACT_GELU_TANH, "FF1 (bias+GELU-tanh, fp16 out)", depth),
            run(3 * D, D, ops.EPI_QKV_ROPE, ops.ACT_NONE, "QKV (bias+RoPE)", depth, seq=seq,
                rope=ops.rope_tables(seq, dev), inner=D, pe_heads=1),
            run(D, D, ops.EPI_RESID, ops.ACT_NONE, "out-proj (gate, TMA reduce-add)", depth),
            run(D, F, ops.EPI_RESID, ops.ACT_NONE, "FF2 (gate, TMA reduce-add)", depth)]
    qkv = [torch.randn(M, 3 * D, generator=g).half().to(dev) for _ in range(3)]
    us = _graph_time_us(lambda: [ops.attention(qkv[i % 3], Be, seq, H) for i in range(12)], 12)
    q4 = [x.view(Be, seq, 3, H, 64).permute(2, 0, 3, 1, 4) for x in qkv]  # [3][Be, H, seq, 64] strided views
    lib = _graph_time_us(lambda: [TF.scaled_dot_product_attention(q4[i % 3][0], q4[i % 3][1], q4[i % 3][2])
                                  for i in range(12)], 12)
    afl = 4.0 * Be * H * seq * seq * 64
    rows.append(dict(kernel="attention (dh 64, non-causal)", shape=[Be, seq, H], launches_per_step=depth,
                     us_per_launch=round(us, 2), tflops=round(afl / us / 1e6, 1), frac=round(afl / us / 1e6 / peaks["tf"], 4),
                     flops_per_launch=afl, library_ref_us=round(lib, 2),
                     library_ref="F.scaled_dot_product_attention fp16 (the reference's call, modules.py:519)"))
    gemms = rows[:4]
    t_gemm = sum(r["us_per_launch"] * r["launches_per_step"] for r in gemms)
    gw = sum(r["frac"] * r["us_per_launch"] * r["launches_per_step"] for r in gemms) / t_gemm
    top = max(rows, key=lambda r: r["us_per_launch"] * r["launches_per_step"])
    traffic = load_traffic()
    tkey = "attention_dram_bytes_per_launch" if top["kernel"].startswith("attention") else "gemm_dram_bytes_per_launch"
    name = ("attn_fwd_tcgen05_kernel" if top["kernel"].startswith("attention")
            else f"gemm_tcgen05_kernel<tile {top['tile']}> ({top['kernel']})")
    return dict(bound="tensor", kernel=name, shape=top["shape"], us_per_launch=top["us_per_launch"],
                achieved=top["tflops"], peak=peaks["tf"], unit="TFLOP/s", frac=top["frac"],
                share_basis="largest us_per_launch x launches_per_step among the kernels below",
                peak_source=peaks["src"] + " bf16_tflops (burst)", flops_per_launch=top["flops_per_launch"],
                traffic=traffic.get(tkey), traffic_source=traffic.get("source"),
                gemm_time_weighted_frac=round(gw, 4), kernels=rows,
                method=">= 192 MB of distinct weights per shape (> L2) launched back to back from a CUDA graph, CUDA events")


def bandwidth_kernels(model, voc, w, peaks, dev):
    """Achieved GB/s of the HBM/L2-bound kernels on their ALGORITHMIC bytes (DESIGN.md §4), CUDA-graph timed."""
    from f5_tts_b200 import ops

    out = []
    g = torch.Generator().manual_seed(5)
    hbm = peaks["hbm"]

    def add(name, us, nbytes, note):
        out.append(dict(kernel=name, us_per_launch=round(us, 2), algorithmic_bytes=int(nbytes),
                        gbs=round(nbytes / us / 1e3, 1), frac_of_hbm=round(nbytes / us / 1e3 / hbm, 4), note=note))

    B = 8
    nw = 282 * 256
    wavs = [(0.1 * torch.randn(B, nw, generator=g)).to(dev) for _ in range(4)]
    us = _graph_time_us(lambda: [model.mel_spec(wavs[i % 4], frames_last=False) for i in range(8)], 8)
    T = 1 + nw // 256
    add("mel_stft_kernel (8 x 3 s)", us, B * (4 * nw + 400 * T), "read 4*nw, write 400*frames (real-input FFT in smem)")
    M, D = 2 * max(w["frames"]), 1024
    xs = [torch.randn(M, D, generator=g).to(dev) for _ in range(3)]
    a, b = torch.randn(D, generator=g).to(dev), torch.randn(D, generator=g).to(dev)
    us = _graph_time_us(lambda: [ops.row_norm(xs[i % 3], 0, a, b) for i in range(12)], 12)
    add(f"row_norm_kernel<0> ({M} x {D})", us, M * D * 6, "read fp32 x, write fp16; operands L2-resident at this size")
    mels = [(torch.randn(B, 100, 656, generator=g) * 1.5 - 2.0).to(dev) for _ in range(3)]
    for m in mels:  # the decode is one CUDA graph inside the library: time its launches directly
        voc.decode(m)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(9):
        voc.decode(mels[i % 3])
    e1.record()
    torch.cuda.synchronize()
    add("vocos decode (8 x 656 frames, whole graph: 30 kernels)", e0.elapsed_time(e1) * 1e3 / 9,
        B * (400 * 656 + 1024 * 655) + 54_000_000 // 2,
        "im2col, 18 GEMMs, dwconv+LN x8, ISTFT: reads mel + fp16 weights once, writes audio; latency-bound")
    return out


def host_cores():
    """(usable cores, torch threads): honours the cgroup CPU quota (the GPU box shows 128 CPUs but grants 16 cores;
    oversubscribing it made the fp32 oracle 50x slower) and the affinity mask."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(round(int(quota) / int(period)))))
    except Exception:  # noqa: BLE001
        pass
    return n, n


class CpuOracle:
    """CPU oracle (port of the reference, fp32) on all granted host cores.  Built once (1.3 GB of synthetic weights, one
    untimed warm-up).  `run(n)` executes the whole hot path with n NFE steps and returns its wall time."""

    def __init__(self, w):
        from oracle import f5_oracle as O

        self.O, self.w = O, w
        self.cores, self.threads = host_cores()
        torch.set_num_threads(self.threads)
        self.cfg = getattr(SD, w["arch"])()
        self.sd = SD.synthetic_state_dict(self.cfg, seed=1234)
        self.vsd = SD.synthetic_vocos_state_dict()
        self.wav, self.text, self.duration, self.lens = synth_inputs(w)
        self.gen = sum(f - r for f, r in zip(w["frames"], w["ref"]))
        self.run(1)  # untimed warm-up: thread pool, oneDNN primitive caches, first touch of the weights

    def run(self, n):
        O, w = self.O, self.w
        t0 = time.perf_counter()
        if w["B"] == 1:
            res = O.sample(self.sd, self.cfg, self.wav, self.text, int(self.duration[0]), steps=n,
                           cfg_strength=CFG_STRENGTH, sway_sampling_coef=SWAY, seed=0)
            ref = self.wav.shape[-1] // 256
        else:
            cond = O.mel_spectrogram(self.wav).permute(0, 2, 1)
            res = O.sample(self.sd, self.cfg, cond, self.text, self.duration, lens=self.lens, steps=n,
                           cfg_strength=CFG_STRENGTH, sway_sampling_coef=SWAY, seed=0)
            ref = int(self.lens.min())
        O.vocos_decode(self.vsd, res.out[:, ref:, :].permute(0, 2, 1))
        return time.perf_counter() - t0

    def full_pass(self):
        """ONE complete pass at the workload's NFE, timed in full — no extrapolation."""
        t = self.run(self.w["nfe"])
        return dict(value=self.gen / t, unit="mel_frames/s", cores=self.cores, threads=self.threads, kind="port",
                    sample=f"one complete pass of the workload (NFE {self.w['nfe']}) through oracle/f5_oracle.py, fp32, "
                           f"{self.threads} threads: {t:.1f} s, timed in full",
                    seconds=t, rtf=t / (self.gen * 256 / 24000.0))


def reference_arm(args, w, config, gen_frames):
    """--impl reference: the reference's CPU path (the pinned oracle PORT of it, `kind: "port"` — the reference modules
    themselves cannot be imported on the GPU box).  Every one of the W + K steps is executed and timed as it is reported:
    a step is a BOUNDED SAMPLE of the workload — the complete hot path (mel, text embedding, sampler, vocoder) with b of
    the workload's NFE solver steps, b sized for ~6 s per step so the run stays within a few minutes — and `value` =
    (generated frames x b / NFE) / step time, i.e. frame-steps per second normalised to the workload's NFE.  One complete
    pass at the full NFE is timed once in the same run (`full_pass`) as the cross-check of that normalisation."""
    oracle = CpuOracle(w)
    t1 = oracle.run(1)
    b = max(2, min(w["nfe"], int(6.0 / max(t1, 1e-3))))
    times = []
    for i in range(args.warmup + args.steps):
        t = oracle.run(b)
        if i >= args.warmup:
            times.append(t)
    t_step = statistics.mean(times)
    v = gen_frames * (b / w["nfe"]) / t_step
    full = oracle.full_pass() if w["B"] == 1 else None
    sample = (f"{b} of {w['nfe']} NFE per step through the whole hot path, every step executed and timed "
              f"({t_step:.2f} s/step); value = generated frames x {b}/{w['nfe']} / step time")
    line = dict(metric="mel_frames_per_sec", value=v, unit="mel_frames/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * t_step, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="fp32", data="synthetic", config=config, impl="reference",
                rtf=(gen_frames / v) / (gen_frames * 256 / 24000.0),
                cpu_baseline=dict(value=v, unit="mel_frames/s", cores=oracle.cores, kind="port", sample=sample),
                full_pass=full,
                e2e=dict(value=v, unit="mel_frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


def parity_vs_reference(model, dev):
    """Same-run parity of the sampler on the headline workload against the unmodified fp32 reference's committed output."""
    import numpy as np

    if not os.path.exists(GOLDEN_CFG2):
        return None
    z = np.load(GOLDEN_CFG2)
    w = WORKLOADS["cfg2"]
    wav, text, duration, _ = synth_inputs(w)
    out, traj = model.sample(wav.to(dev), text.to(dev), int(duration[0]), steps=int(z["steps"]), cfg_strength=CFG_STRENGTH,
                             sway_sampling_coef=SWAY, seed=0, y0=torch.from_numpy(z["y0"]).to(dev))
    n_ref = int(z["n_ref"])

    def rel(a, b):
        a, b = a.float().cpu(), torch.from_numpy(b)
        return float((a[:, n_ref:] - b[:, n_ref:]).norm() / b[:, n_ref:].norm())

    kept = [int(k) for k in z["kept"]]
    drift = {str(k): round(rel(traj[k], z[f"traj_{k}"]), 6) for k in kept}
    return dict(rel_l2=drift[str(kept[-1])], gate=5e-3, steps=int(z["steps"]), region="generated frames of the final mel",
                vs="tests/golden/cfg2_full_nfe32.npz: unmodified reference CFM.sample, fp32 CPU, same weights / inputs / y0",
                drift_per_step=drift,
                reference_fp16_drift_per_step={str(k): round(float(v), 6) for k, v in zip(kept, z["ref_fp16_drift"])},
                passed=bool(all(v <= 5e-3 for v in drift.values())))


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each tensor as out_dir/<name>.npy in float32 (every workload's outputs fit DUMP_LIMIT whole)."""
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def timed(fn, steps, warmup, barrier):
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / steps


def extra_workloads(dev, world, rank, dist, barrier, models):
    """cfg3 / cfg5 on one GPU (rank 0's GPU; every rank runs them so the ranks stay in step) and the sharded cfg4."""
    from f5_tts_b200 import sharding

    recs = []

    def reduce_max(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    if world == 1:
        for name in ("cfg3", "cfg5"):
            w = WORKLOADS[name]
            model, voc = models(w["arch"])
            wav, text, duration, lens = (t.to(dev) for t in synth_inputs(w))
            ms = timed(lambda: hot_path(model, voc, wav, text, duration, lens, w["nfe"]), 3, 2, barrier)
            gen = sum(f - r for f, r in zip(w["frames"], w["ref"]))
            flops = model.transformer.sample_flops(w["B"], max(w["frames"]), w["nfe"], CFG_STRENGTH)
            recs.append(dict(workload=name, arch=w["arch"], batch=w["B"], frames=w["frames"], nfe=w["nfe"], n_gpus=1,
                             ms_per_step=round(ms, 2), value=round(gen / (ms * 1e-3), 1), unit="mel_frames/s",
                             rtf=round(ms * 1e-3 / (gen * 256 / 24000.0), 5), steps=3, warmup=2,
                             step_tflops=round(flops / (ms * 1e-3) / 1e12, 1),
                             mode="faithful (padded rows computed and attended, as the reference's batched call)"))
        # cfg3 again in packed / variable-length execution (SURVEY.md §8f-1): every utterance exactly as if alone in the
        # batch — keys masked, padded tiles skipped (the reference's counterpart is its masked / varlen mode)
        w = WORKLOADS["cfg3"]
        model, voc = models(w["arch"])
        wav, text, duration, lens = (t.to(dev) for t in synth_inputs(w))
        ms = timed(lambda: hot_path(model, voc, wav, text, duration, lens, w["nfe"], exact_varlen=True), 3, 2, barrier)
        gen = sum(f - r for f, r in zip(w["frames"], w["ref"]))
        recs.append(dict(workload="cfg3", arch=w["arch"], batch=w["B"], frames=w["frames"], nfe=w["nfe"], n_gpus=1,
                         ms_per_step=round(ms, 2), value=round(gen / (ms * 1e-3), 1), unit="mel_frames/s",
                         rtf=round(ms * 1e-3 / (gen * 256 / 24000.0), 5), steps=3, warmup=2,
                         mode="exact_varlen (keys masked per utterance, tiles that hold only padding skipped)"))
        # one request of several text chunks through infer_batch_process: ONE batched sampler call (exact_varlen, shared
        # prompt mel, device-side cross-fade) against the reference's structure, one sampler call per chunk
        from f5_tts_b200 import infer as INF

        w2 = WORKLOADS["cfg2"]
        model, voc = models(w2["arch"])
        audio_h = synth_inputs(w2)[0].clone().pin_memory()
        ref_text = "some call me nature others call me mother na."
        base = "i have been a silent spectator watching species evolve and empires rise and fall but always remember i am mighty"
        chunks = [base[:100] + ".", base[:70] + ".", base[:90] + ".", base[:60] + "."]
        kw = dict(nfe_step=w2["nfe"], cfg_strength=CFG_STRENGTH, sway_sampling_coef=SWAY, device=dev)

        def batched():
            return next(INF.infer_batch_process((audio_h, 24000), ref_text, chunks, model, voc, **kw))

        def per_chunk():
            return [next(INF.infer_batch_process((audio_h, 24000), ref_text, [c], model, voc, **kw)) for c in chunks]

        frames = batched()[2].shape[-1]
        ms_b = timed(batched, 3, 1, barrier)
        ms_s = timed(per_chunk, 3, 1, barrier)
        recs.append(dict(workload="chunked request (4 text chunks, 10 s prompt-conditioned each, NFE 32) through infer_batch_process",
                         generated_frames=int(frames), n_gpus=1, steps=3, warmup=1,
                         batched_ms=round(ms_b, 2), per_chunk_ms=round(ms_s, 2), speedup=round(ms_s / ms_b, 3),
                         value=round(frames / (ms_b * 1e-3), 1), unit="mel_frames/s",
                         note="host audio in, host waveform out; batched = one exact_varlen sampler call for all chunks"))
        # request-level serving (Triton Python backend mirror, serving.py): 4 requests with different reference lengths
        # and texts through ONE execute() (max_batch_size 4, as config.pbtxt) against one execute() per request
        from f5_tts_b200 import serving as SRV

        proc = SRV.F5TTSRequestProcessor(model, voc, device=dev, nfe_step=w2["nfe"])
        wav_np = synth_inputs(w2)[0].numpy()
        reqs = [dict(reference_wav=wav_np[:, : 24000 * s], reference_wav_len=np.array([24000 * s], np.int32),
                     reference_text=ref_text[: 15 * s], target_text=(base + " " + base)[: 35 * s * k])
                for s, k in ((3, 2), (2, 3), (3, 1), (2, 2))]
        outs = proc.execute(reqs)
        audio_s = sum(len(o) for o in outs) / 24000.0
        ms_b = timed(lambda: proc.execute(reqs), 3, 1, barrier)
        ms_s = timed(lambda: [proc.execute([r]) for r in reqs], 3, 1, barrier)
        recs.append(dict(workload="serving: 4 requests (2-3 s reference, 7-14 s generated, NFE 32) through "
                                  "serving.F5TTSRequestProcessor.execute (Triton Python backend contract)",
                         generated_audio_s=round(audio_s, 2), n_gpus=1, steps=3, warmup=1, batched_ms=round(ms_b, 2),
                         per_request_ms=round(ms_s, 2), speedup=round(ms_s / ms_b, 3), rtf=round(ms_b * 1e-3 / audio_s, 5),
                         note="host numpy in, host numpy out; the reference publishes RTF 0.0394 for this contract on an "
                              "L20 with TensorRT-LLM (other hardware, other prompts: not a baseline for vs_baseline)"))
    # cfg4: 64 fixed 10 s utterances, NFE 16, sharded by utterance over the ranks; batches of 8 per sampler call
    w = WORKLOADS["cfg4"]
    model, voc = models(w["arch"])
    n_utt = 64
    durations = [w["frames"][0]] * n_utt
    mine = sharding.plan_shards(durations, world)[rank]
    g = torch.Generator().manual_seed(11)
    wav_all = 0.1 * torch.randn(n_utt, w["ref"][0] * 256, generator=g)
    text_all = torch.randint(0, 2545, (n_utt, w["nt"]), generator=g)
    idx = torch.tensor(mine, dtype=torch.long)
    wav_d, text_d = wav_all[idx].to(dev), text_all[idx].to(dev)
    lens_d = torch.full((len(mine),), w["ref"][0], dtype=torch.long, device=dev)
    dur_d = torch.full((len(mine),), w["frames"][0], dtype=torch.long, device=dev)

    def sharded_pass():
        mels, auds = [], []
        for s in range(0, len(mine), 8):
            m, a = hot_path(model, voc, wav_d[s:s + 8], text_d[s:s + 8], dur_d[s:s + 8], lens_d[s:s + 8], w["nfe"])
            mels.append(m[:, w["ref"][0]:])
            auds.append(a)
        mel, aud = torch.cat(mels), torch.cat(auds)
        if dist is not None:  # ONE padded all-gather of the finished mel + audio (sharding.gather_padded, NCCL)
            n = torch.full((mel.shape[0],), mel.shape[1], dtype=torch.int64, device=dev)
            sharding.gather_padded(mel, n)
            sharding.gather_padded(aud.unsqueeze(-1), n * 256)

    ms = reduce_max(timed(sharded_pass, 2, 1, barrier))
    gen = n_utt * (w["frames"][0] - w["ref"][0])
    recs.append(dict(workload="cfg4", arch=w["arch"], batch=n_utt, per_gpu=len(mine), frames=w["frames"][0], nfe=w["nfe"],
                     n_gpus=world, scaling="strong", ms_per_step=round(ms, 2), value=round(gen / (ms * 1e-3), 1),
                     unit="mel_frames/s", rtf=round(ms * 1e-3 / (gen * 256 / 24000.0), 6), steps=2, warmup=1,
                     parallelism=f"plan_shards: {n_utt} utterances over {world} rank(s), batches of 8, "
                                 "one padded all-gather of mel + audio at the end (no collective inside the NFE loop)"))
    return recs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg3/cfg4/cfg5 records and the per-kernel tables")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0's mel and audio) as "
                         "DIR/<name>.npy in float32; the inputs are seeded, so two builds can be compared output by output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    gen_frames = sum(f - r for f, r in zip(w["frames"], w["ref"]))
    config = dict(workload=f"{args.workload}: {w['arch']} B={w['B']}/GPU frames={w['frames'] if w['B'] > 1 and len(set(w['frames'])) > 1 else w['frames'][0]} "
                           f"prompt={w['ref'][0] if len(set(w['ref'])) == 1 else w['ref']} NFE={w['nfe']} cfg={CFG_STRENGTH} sway={SWAY}",
                  global_batch=w["B"] * max(world, 1), parallelism=f"dp{world} (utterance sharding, all-gather of mel+audio per step)",
                  l2="no explicit flush: each step streams 0.67 GB of fp16 weights (> 126 MB L2)")

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, w, config, gen_frames)
        return

    assert torch.cuda.is_available(), "bench.py --impl b200 needs a CUDA (B200) device; there is no CPU fallback"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    from f5_tts_b200 import _lib
    from f5_tts_b200 import infer as INF

    peaks = load_peaks()
    _models = {}

    def models(arch):
        if arch not in _models:
            _models[arch] = build_gpu_model(arch, dev)
        return _models[arch][0], _models[arch][1]

    model, voc = models(w["arch"])
    cfg = _models[w["arch"]][2]
    wav, text, duration, lens = synth_inputs(w)
    wav_d, text_d, dur_d, lens_d = wav.to(dev), text.to(dev), duration.to(dev), lens.to(dev)
    nfe = w["nfe"]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def gather(mel, audio):
        if dist is None:
            return
        m = torch.empty((world * mel.shape[0],) + tuple(mel.shape[1:]), device=dev, dtype=mel.dtype)
        a = torch.empty((world * audio.shape[0],) + tuple(audio.shape[1:]), device=dev, dtype=audio.dtype)
        dist.all_gather_into_tensor(m, mel.contiguous())
        dist.all_gather_into_tensor(a, audio.contiguous())

    # ---- device-resident throughput -------------------------------------------------------------------------
    for _ in range(args.warmup):
        gather(*hot_path(model, voc, wav_d, text_d, dur_d, lens_d, nfe, w['frames'][0]))
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as cs:
        barrier()
        e0.record()
        for _ in range(args.steps):
            last = hot_path(model, voc, wav_d, text_d, dur_d, lens_d, nfe, w['frames'][0])
            gather(*last)
        e1.record()
        barrier()
    launches = _lib.launch_count() - l0
    ms = e0.elapsed_time(e1) / args.steps
    clocks = cs.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("mel", "audio"), last)))

    # ---- end to end through the reference-facing call with HOST buffers ---------------------------------------
    if w["B"] == 1:
        # infer_process((audio, sr), ref_text, gen_text, ...): host audio in, host numpy waveform out.  The text is
        # sized so that the call does exactly the workload: 150 tokens, fix_duration -> 938 frames, one chunk.
        n_ref_txt = 45
        ref_text = ("some call me nature others call me mother na" + ".")[:n_ref_txt - 1] + "."
        gen_text = ("i have been a silent spectator watching species evolve and empires rise and fall but always remember "
                    "i am mighty")[: w["nt"] - n_ref_txt - 1]
        fix_dur = (w["frames"][0] + 0.25) * 256 / 24000.0
        audio_h = wav.clone().pin_memory()  # [1, nw] host
        h2d = audio_h.numel() * 4 + w["nt"] * 8
        d2h = 256 * (w["frames"][0] - w["ref"][0] - 1) * 4

        def e2e_step():
            wave_np, sr, spec = INF.infer_process((audio_h, 24000), ref_text, gen_text, model, voc, nfe_step=nfe,
                                                  cfg_strength=CFG_STRENGTH, sway_sampling_coef=SWAY, fix_duration=fix_dur,
                                                  device=dev, show_info=lambda *_: None)
            assert spec.shape[-1] == w["frames"][0] - w["ref"][0] and len(wave_np) * 4 == d2h
        e2e_api = "f5_tts_b200.infer.infer_process (utils_infer.py:384-434 mirror): host audio -> host waveform"
    else:
        wav_h, text_h = wav.pin_memory(), text.pin_memory()
        n_audio = 256 * (max(w["frames"]) - min(w["ref"]) - 1)
        out_h = torch.empty((w["B"], n_audio), dtype=torch.float32).pin_memory()
        h2d, d2h = wav.numel() * 4 + text.numel() * 8, out_h.numel() * 4

        def e2e_step():
            wd, td = wav_h.to(dev, non_blocking=True), text_h.to(dev, non_blocking=True)
            _, audio = hot_path(model, voc, wd, td, dur_d, lens_d, nfe, w['frames'][0])
            out_h.copy_(audio, non_blocking=True)
            torch.cuda.current_stream().synchronize()  # the caller holds the waveform on the host here
        e2e_api = "CFM.sample + Vocos.decode with pinned host buffers"

    for _ in range(args.warmup):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(args.steps):
        e2e_step()
    g1.record()
    barrier()
    ms_e2e = max(g0.elapsed_time(g1), (time.perf_counter() - t0) * 1e3) / args.steps

    # ---- max over ranks --------------------------------------------------------------------------------------
    if dist is not None:
        tt = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(tt[0]), float(tt[1])
    total_frames = gen_frames * world
    value = total_frames / (ms * 1e-3)
    e2e_value = total_frames / (ms_e2e * 1e-3)
    audio_sec = gen_frames * 256 / 24000.0

    extras = [] if args.no_extras else extra_workloads(dev, world, rank, dist, barrier, models)

    if rank == 0:
        flops = model.transformer.sample_flops(w["B"], max(w["frames"]), nfe, CFG_STRENGTH)
        step_tf = flops / (ms * 1e-3) / 1e12
        step_tensor = dict(flops_per_step=flops, achieved=round(step_tf, 1), peak=peaks["tf_sus"], unit="TFLOP/s",
                           frac=round(step_tf / peaks["tf_sus"], 4),
                           note="whole hot-path step (all kernels, launch gaps included) vs sustained bf16 peak")
        if args.no_extras:
            roof = dict(bound="tensor", step_tensor=step_tensor)
        else:
            seq = max(w["frames"]) + (1 if cfg.backbone == "UNetT" else 0)
            roof = isolated_kernel_roofline(cfg, 2 * w["B"] * seq, seq, peaks, dev)
            roof["step_tensor"] = step_tensor
            roof["bandwidth_kernels"] = bandwidth_kernels(model, voc, w, peaks, dev)
        parity = parity_vs_reference(model, dev) if args.workload == "cfg2" else None
        cpu = None
        if not (args.no_cpu_baseline or world > 1):  # timed at N = 1 only
            cpu = CpuOracle(w).full_pass() if w["B"] == 1 else None
        line = dict(metric="mel_frames_per_sec", value=value, unit="mel_frames/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="fp16 operands / fp32 accumulate+state", data="synthetic (random-init weights, released checkpoint layout)",
                    config=config, rtf=(ms * 1e-3) / audio_sec, rtf_e2e=(ms_e2e * 1e-3) / audio_sec,
                    e2e=dict(value=e2e_value, unit="mel_frames/s", ms_per_step=ms_e2e, api=e2e_api,
                             h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h),
                    gpu_launches=int(launches), parity=parity, roofline=roof, workloads=extras, cpu_baseline=cpu,
                    clocks=clocks, impl="b200")
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
