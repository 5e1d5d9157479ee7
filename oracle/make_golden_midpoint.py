"""Golden vectors of the midpoint ODE solver (odeint_kwargs=dict(method="midpoint"), cfm.py:39-42) — TEST INFRASTRUCTURE.

    python oracle/make_golden_midpoint.py             # all seven fixtures (~12 min on 8 cores, mostly cfg3)
    python oracle/make_golden_midpoint.py reference   # only the five written by the reference (~1 min)
    python oracle/make_golden_midpoint.py fullsize    # only the two full-size oracle fixtures

* Reference fixtures (same format as oracle/make_golden.py's, plus `method`): the UNMODIFIED reference modules, imported
  with the torchdiffeq midpoint restatement of oracle/ode_midpoint.py, on seeded synthetic weights and inputs; the
  oracle's result on the same inputs is printed next to it (rel-L2 0.0 at generation time).  Two tiny DiT cases for the
  CPU oracle check and three base-width cases mirroring f5base_b1_n192 / f5v1base_b1_n128 / e2base_b1_n128 for the GPU.
* Full-size fixtures (same format as oracle/make_golden_fullsize.py's, plus `method`): the CPU oracle at the cfg2 shape
  on the EPSS-16 grid (32 evaluations, the cost of Euler NFE 32) and at the cfg3 masked shape with 4 steps.  cfg3 keeps
  every 12th generated row of every utterance (cfg2 every 3rd), which keeps the file small.
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import synthdata as SD  # noqa: E402
from oracle import f5_oracle as O  # noqa: E402
from oracle import ode_midpoint as M  # noqa: E402
from oracle.make_golden import rel_l2, tiny_dit  # noqa: E402
from oracle.make_golden_fullsize import draw_y0  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
METHOD = "midpoint"


def reference_case(name, cfg, *, B, n_ref, nt, durations, lens=None, steps, cfg_strength, sway, seed, wseed=1234,
                   text_pad=None):
    t0 = time.time()
    cfm, dit, unett, _, _ = M.import_reference()
    sd = O.synthetic_state_dict(cfg, seed=wseed)
    kw = dict(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, dim_head=cfg.dim_head, ff_mult=cfg.ff_mult,
              mel_dim=cfg.mel_dim, text_num_embeds=cfg.text_num_embeds, text_dim=cfg.text_dim,
              text_mask_padding=cfg.text_mask_padding, conv_layers=cfg.conv_layers, pe_attn_head=cfg.pe_attn_head,
              attn_backend="torch", attn_mask_enabled=cfg.attn_mask_enabled)
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        backbone = (dit.DiT if cfg.backbone == "DiT" else unett.UNetT)(**kw)
    model = cfm.CFM(transformer=backbone,
                    mel_spec_kwargs=dict(n_fft=1024, hop_length=256, win_length=1024, n_mel_channels=100,
                                         target_sample_rate=24000, mel_spec_type="vocos"),
                    odeint_kwargs=dict(method=METHOD), vocab_char_map=None)
    res = model.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    model.eval()
    g = torch.Generator().manual_seed(100 + seed)
    cond = torch.randn(B, n_ref, 100, generator=g)
    text = torch.randint(0, cfg.text_num_embeds, (B, nt), generator=g)
    if text_pad is not None:
        for b, keep in enumerate(text_pad):
            text[b, keep:] = -1
    duration = durations if isinstance(durations, int) else torch.tensor(durations, dtype=torch.long)
    lens_t = None if lens is None else torch.tensor(lens, dtype=torch.long)
    with torch.no_grad():
        out, traj = model.sample(cond=cond, text=text, duration=duration, lens=lens_t, steps=steps,
                                 cfg_strength=cfg_strength, sway_sampling_coef=sway, seed=seed)
    ora = M.sample(sd, cfg, cond, text, duration, lens=lens_t, steps=steps, cfg_strength=cfg_strength,
                   sway_sampling_coef=sway, seed=seed, method=METHOD)
    print(f"[{name}] ref out {tuple(out.shape)} oracle-vs-ref rel-L2 {rel_l2(ora.out, out):.3e}  ({time.time() - t0:.1f}s)",
          flush=True)
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), cond=cond.numpy(), text=text.numpy(),
                        duration=np.asarray(durations), lens=np.asarray(lens if lens is not None else []),
                        steps=steps, cfg_strength=cfg_strength, sway=np.asarray(np.nan if sway is None else sway),
                        seed=seed, wseed=wseed, out=out.numpy(), y0=traj[0].numpy(), traj_last=traj[-1].numpy(),
                        traj_1=traj[1].numpy(), cfg=np.asarray(repr(cfg)), method=np.asarray(METHOD))


def reference_goldens():
    reference_case("dit_tiny_b1_midpoint", tiny_dit(), B=1, n_ref=20, nt=24, durations=64, steps=3, cfg_strength=2.0,
                   sway=-1.0, seed=3)
    reference_case("dit_tiny_b3_midpoint", tiny_dit(), B=3, n_ref=30, nt=40, durations=[90, 64, 77],
                   lens=[30, 18, 25], steps=3, cfg_strength=2.0, sway=-1.0, seed=5, text_pad=[40, 25, 33])
    reference_case("f5base_b1_n192_midpoint", O.f5tts_base(), B=1, n_ref=58, nt=31, durations=192, steps=3,
                   cfg_strength=2.0, sway=-1.0, seed=0)
    reference_case("f5v1base_b1_n128_midpoint", O.f5tts_v1_base(), B=1, n_ref=40, nt=20, durations=128, steps=2,
                   cfg_strength=2.0, sway=-1.0, seed=2)
    reference_case("e2base_b1_n128_midpoint", O.e2tts_base(), B=1, n_ref=40, nt=20, durations=128, steps=2,
                   cfg_strength=2.0, sway=-1.0, seed=2, wseed=99)


FULLSIZE = {
    # name: (arch factory, attn_mask_enabled, workload, solver steps, row stride)
    "cfg2_midpoint16": ("f5tts_base", False, "cfg2", 16, 3),
    "cfg3_masked_midpoint4": ("f5tts_base", True, "cfg3", 4, 12),
}


def fullsize_goldens():
    for name, (arch, attn_mask, wl, steps, stride) in FULLSIZE.items():
        cfg = getattr(SD, arch)()
        cfg.attn_mask_enabled = attn_mask
        w = SD.WORKLOADS[wl]
        sd = SD.synthetic_state_dict(cfg, seed=1234)
        wav, text, duration, lens = SD.synth_inputs(w)
        cond = O.mel_spectrogram(wav).permute(0, 2, 1).contiguous()
        y0 = draw_y0(duration, cfg.mel_dim, seed=0)
        t0 = time.time()
        ref = M.sample(sd, cfg, cond, text, duration, lens=lens, steps=steps, cfg_strength=SD.CFG_STRENGTH,
                       sway_sampling_coef=SD.SWAY, seed=0, y0=y0, method=METHOD)

        def kept(t):
            return torch.cat([t[b, int(lens[b]): int(duration[b]): stride] for b in range(t.shape[0])], 0)

        path = os.path.join(GOLD, f"fullsize_{name}.npz")
        np.savez(path, stride=stride, steps=steps, wseed=1234, seed=0, arch=arch, attn_mask_enabled=attn_mask,
                 workload=wl, method=METHOD,
                 y0_checksum=np.array([float(y0.double().sum()), float(y0.double().abs().sum())]),
                 step1=kept(ref.trajectory[1]).numpy(), final=kept(ref.out).numpy())
        print(f"{name}: {steps} steps in {time.time() - t0:.0f} s, {os.path.getsize(path) / 1e6:.2f} MB", flush=True)


def main():
    torch.set_num_threads(os.cpu_count() or 8)
    which = sys.argv[1:] or ["reference", "fullsize"]
    if "reference" in which:
        reference_goldens()
    if "fullsize" in which:
        fullsize_goldens()


if __name__ == "__main__":
    main()
