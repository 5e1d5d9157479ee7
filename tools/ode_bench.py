"""Solver cost and accuracy at equal backbone evaluations on the cfg2 workload (F5-TTS Base, B=1, 938 frames,
CFG 2, sway -1): Euler NFE 32, midpoint 16 steps (the same 32 evaluations, EPSS-16 grid) and midpoint 32 steps.

    python tools/ode_bench.py [--rounds 10] [--warmup 2] [--out profiles/ode_midpoint_cfg2.txt]

One process; the arms alternate within every round so that clock and neighbour drift hits them alike.  Per arm:
device time of one CFM.sample call (CUDA events, after warm-up; median and min..max over rounds), that time per
backbone evaluation, and the rel-L2 of the generated mel against a midpoint run with 64 steps of the same engine
(the solver's error at that cost).  Sampling only: the prompt mel is computed once, the vocoder is not run.
Prints the card name and power limit next to the numbers.
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import f5_tts_b200 as F5  # noqa: E402
import synthdata as SD  # noqa: E402

ARMS = [("euler", 32), ("midpoint", 16), ("midpoint", 32)]
REFERENCE = ("midpoint", 64)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", help="also write the report to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "ode_bench.py times the B200 engine: it needs a CUDA device"
    dev = "cuda:0"
    w = SD.WORKLOADS["cfg2"]
    cfg = SD.f5tts_base()
    tr = F5.DiT(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, ff_mult=cfg.ff_mult, text_dim=cfg.text_dim,
                text_mask_padding=cfg.text_mask_padding, conv_layers=cfg.conv_layers, pe_attn_head=cfg.pe_attn_head,
                text_num_embeds=cfg.text_num_embeds, mel_dim=100)
    base = F5.CFM(transformer=tr)
    base.load_state_dict(SD.synthetic_state_dict(cfg, seed=1234), strict=True)
    base = base.to(dev)
    models = {m: F5.CFM(transformer=base.transformer, odeint_kwargs=dict(method=m)).to(dev) for m in ("euler", "midpoint")}
    wav, text, duration, _ = SD.synth_inputs(w)
    cond = base.mel_spec(wav.to(dev), frames_last=False)
    text, frames, n_ref = text.to(dev), int(duration[0]), w["ref"][0]

    def call(method, steps):
        out, _ = models[method].sample(cond, text, frames, steps=steps, cfg_strength=SD.CFG_STRENGTH,
                                       sway_sampling_coef=SD.SWAY, seed=0)
        return out

    ref = call(*REFERENCE)[:, n_ref:].float()
    outs, times = {}, {a: [] for a in ARMS}
    for a in ARMS:
        for _ in range(args.warmup):
            outs[a] = call(*a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for a in ARMS:
            e0.record()
            out = call(*a)
            e1.record()
            e1.synchronize()
            times[a].append(e0.elapsed_time(e1))
            assert torch.equal(out, outs[a]), f"{a}: not bit-identical run to run"
    lines = [f"card: {card()}",
             f"workload: cfg2 (F5-TTS Base, B=1, {frames} frames, prompt {n_ref}, CFG {SD.CFG_STRENGTH}, sway {SD.SWAY}); "
             f"CFM.sample only, {args.rounds} alternating rounds after {args.warmup} warm-up calls per arm",
             f"solver error: rel-L2 of the generated mel rows against {REFERENCE[0]} {REFERENCE[1]} steps, same engine",
             f"{'arm':<16}{'evals':>6}{'ms/call median':>16}{'(min..max)':>18}{'ms/eval':>9}{'rel-L2 vs ref':>15}"]
    for a in ARMS:
        t = sorted(times[a])
        evals = a[1] * (2 if a[0] == "midpoint" else 1)
        med = t[len(t) // 2]
        err = float((outs[a][:, n_ref:].float() - ref).norm() / ref.norm())
        lines.append(f"{a[0] + ' ' + str(a[1]):<16}{evals:>6}{med:>16.2f}{f'({t[0]:.2f}..{t[-1]:.2f})':>18}"
                     f"{med / evals:>9.3f}{err:>15.3e}")
    report = "\n".join(lines)
    print(report)
    if args.out:
        with open(args.out, "w") as f:
            f.write(report + "\n")


if __name__ == "__main__":
    main()
