"""Generate tests/golden/*.npz by running the UNMODIFIED reference (TEST INFRASTRUCTURE).

Run in the build container, where /root/reference exists:

    python -m oracle.make_golden            # writes tests/golden/, prints oracle-vs-reference deltas

The reference modules are imported through oracle/ref_shims.py (third-party stand-ins only);
weights are oracle.f5_oracle.synthetic_state_dict(...) loaded with load_state_dict(strict=True),
which also pins the checkpoint key layout (SURVEY.md §8b).  Every fixture stores the inputs that
cannot be regenerated from a seed alone plus the reference outputs; weights are NOT stored
(regenerated from (config, seed) by tests).  The GPU box has no /root/reference: tests read only
the committed .npz files.
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import f5_oracle as O  # noqa: E402
from oracle import ref_shims  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def tiny_dit(**over) -> O.ArchConfig:
    base = dict(backbone="DiT", dim=128, depth=2, heads=2, dim_head=64, ff_mult=2, mel_dim=100, text_num_embeds=50,
                text_dim=64, text_mask_padding=False, conv_layers=2, pe_attn_head=1, attn_mask_enabled=False)
    base.update(over)
    return O.ArchConfig(**base)


def tiny_unett(**over) -> O.ArchConfig:
    base = dict(backbone="UNetT", dim=128, depth=4, heads=2, dim_head=64, ff_mult=4, mel_dim=100, text_num_embeds=50,
                text_dim=None, text_mask_padding=False, conv_layers=0, pe_attn_head=1, attn_mask_enabled=False)
    base.update(over)
    return O.ArchConfig(**base)


def build_reference(cfg: O.ArchConfig, sd):
    cfm, dit, unett, modules, utils = ref_shims.import_reference()
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
                    odeint_kwargs=dict(method="euler"), vocab_char_map=None)
    missing = model.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return model.eval()


def rel_l2(a, b):
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def run_case(name, cfg, *, B, n_ref, nt, durations, lens=None, steps, cfg_strength, sway, seed, wave=False,
             wseed=1234, text_pad=None):
    t0 = time.time()
    sd = O.synthetic_state_dict(cfg, seed=wseed)
    model = build_reference(cfg, sd)
    g = torch.Generator().manual_seed(100 + seed)
    cond = 0.1 * torch.randn(B, n_ref * 256, generator=g) if wave else torch.randn(B, n_ref, 100, generator=g)
    text = torch.randint(0, cfg.text_num_embeds, (B, nt), generator=g)
    if text_pad is not None:  # ragged text: pad tail with -1 like list_str_to_idx (utils.py:99-106)
        for b, keep in enumerate(text_pad):
            text[b, keep:] = -1
    duration = durations if isinstance(durations, int) else torch.tensor(durations, dtype=torch.long)
    lens_t = None if lens is None else torch.tensor(lens, dtype=torch.long)
    with torch.no_grad():
        out, traj = model.sample(cond=cond, text=text, duration=duration, lens=lens_t, steps=steps,
                                 cfg_strength=cfg_strength, sway_sampling_coef=sway, seed=seed)
    res = O.sample(sd, cfg, cond, text, duration, lens=lens_t, steps=steps, cfg_strength=cfg_strength,
                   sway_sampling_coef=sway, seed=seed)
    d_out = rel_l2(res.out, out)
    d_y0 = float((res.y0 - traj[0]).abs().max())
    print(f"[{name}] ref out {tuple(out.shape)} oracle-vs-ref rel-L2 {d_out:.3e}  y0 max|d| {d_y0:.1e}  "
          f"|out| rms {float(out.pow(2).mean().sqrt()):.3f}  ({time.time() - t0:.1f}s)")
    save = dict(cond=cond.numpy(), text=text.numpy(),
                duration=np.asarray(durations), lens=np.asarray(lens if lens is not None else []),
                steps=steps, cfg_strength=cfg_strength, sway=np.asarray(np.nan if sway is None else sway),
                seed=seed, wseed=wseed, out=out.numpy(), y0=traj[0].numpy(), traj_last=traj[-1].numpy(),
                traj_1=traj[1].numpy(), cfg=np.asarray(repr(cfg)))
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **save)
    return d_out


def per_op_goldens():
    """Outputs of individual reference modules at F5-TTS Base width, small N (kernel-level parity anchors)."""
    cfm, dit, unett, modules, utils = ref_shims.import_reference()
    cfg = O.f5tts_base()
    sd = O.synthetic_state_dict(cfg, seed=1234)
    model = build_reference(cfg, sd)
    tr = model.transformer
    g = torch.Generator().manual_seed(77)
    B, N = 2, 64
    x = torch.randn(B, N, 1024, generator=g)
    t_emb_in = torch.tensor([0.37, 0.37])
    mask = O.lens_to_mask(torch.tensor([64, 45]))
    out = {}
    with torch.no_grad():
        t_emb = tr.time_embed(t_emb_in)
        out["time_embed"] = t_emb.numpy()
        rope = tr.rotary_embed.forward_from_seq_len(N)
        out["rope_freqs"] = rope[0].numpy()
        blk = tr.transformer_blocks[3]
        out["block3_nomask"] = blk(x, t_emb, mask=None, rope=rope).numpy()
        out["block3_mask"] = blk(x, t_emb, mask=mask, rope=rope).numpy()
        norm, gate_msa, shift_mlp, scale_mlp, gate_mlp = blk.attn_norm(x, emb=t_emb)
        out["adaln_norm"] = norm.numpy()
        out["attn_nomask"] = blk.attn(x=norm, mask=None, rope=rope).numpy()
        out["convpos_mask"] = tr.input_embed.conv_pos_embed(x, mask=mask).numpy()
        out["convpos_nomask"] = tr.input_embed.conv_pos_embed(x, mask=None).numpy()
        text = torch.randint(0, 2545, (B, 40), generator=g)
        text[1, 30:] = -1
        out["text_in"] = text.numpy()
        out["text_embed_cond"] = tr.text_embed(text, seq_len=N, drop_text=False).numpy()
        out["text_embed_uncond"] = tr.text_embed(text, seq_len=N, drop_text=True).numpy()
        out["text_embed_cond_varlen"] = tr.text_embed(text, seq_len=mask.sum(dim=1), drop_text=False).numpy()
        out["norm_out"] = tr.norm_out(x, t_emb).numpy()
    out["x"] = x.numpy()
    out["t"] = t_emb_in.numpy()
    # oracle cross-check
    ang = O.rope_angles(N)
    o_blk = O.dit_block(sd, cfg, 3, x, torch.from_numpy(out["time_embed"]), None, ang)
    o_blk_m = O.dit_block(sd, cfg, 3, x, torch.from_numpy(out["time_embed"]), mask, ang)
    print("[per-op] block3 nomask", rel_l2(o_blk, torch.from_numpy(out["block3_nomask"])),
          "mask", rel_l2(o_blk_m, torch.from_numpy(out["block3_mask"])))
    print("[per-op] convpos", rel_l2(O.conv_position_embedding(sd, x, mask), torch.from_numpy(out["convpos_mask"])))
    print("[per-op] text", rel_l2(O.text_embedding_dit(sd, cfg, text, N, False), torch.from_numpy(out["text_embed_cond"])),
          rel_l2(O.text_embedding_dit(sd, cfg, text, mask.sum(dim=1), False),
                 torch.from_numpy(out["text_embed_cond_varlen"])))
    np.savez_compressed(os.path.join(GOLD, "per_op_f5base.npz"), **{k: v.astype(np.float32) if v.dtype.kind == "f" else v
                                                                    for k, v in out.items()})


def mel_golden():
    cfm, dit, unett, modules, utils = ref_shims.import_reference()
    g = torch.Generator().manual_seed(7)
    wav = 0.1 * torch.randn(2, 24000, generator=g)
    ref = modules.MelSpec()(wav)
    mine = O.mel_spectrogram(wav)
    print("[mel] ref", tuple(ref.shape), "oracle max|d|", float((ref - mine).abs().max()))
    np.savez_compressed(os.path.join(GOLD, "mel_vocos.npz"), wav=wav.numpy(), mel=ref.numpy())


def istft_golden():
    g = torch.Generator().manual_seed(9)
    T = 40
    re, im = torch.randn(1, 513, T, generator=g), torch.randn(1, 513, T, generator=g)
    spec = torch.complex(re, im)
    ref = torch.istft(spec, 1024, 256, 1024, torch.hann_window(1024), center=True)
    mine = O.istft_center(spec)
    print("[istft] torch.istft", tuple(ref.shape), "oracle max|d|", float((ref - mine).abs().max()))
    np.savez_compressed(os.path.join(GOLD, "istft_torch.npz"), re=re.numpy(), im=im.numpy(), wav=ref.numpy())


def vocos_golden():
    """No reference implementation exists in the tree or the image (vocos pkg absent): parity unpinned.
    The fixture only freezes the oracle's own output so the CUDA path and later oracle edits are
    compared against a fixed vector."""
    vsd = O.synthetic_vocos_state_dict()
    g = torch.Generator().manual_seed(11)
    mel = torch.randn(1, 100, 64, generator=g) * 1.5 - 2.0
    wav = O.vocos_decode(vsd, mel)
    print("[vocos] oracle-frozen", tuple(wav.shape), "rms", float(wav.pow(2).mean().sqrt()))
    np.savez_compressed(os.path.join(GOLD, "vocos_oracle_frozen.npz"), mel=mel.numpy(), wav=wav.numpy())


def ref_tiny_b2_golden():
    """Batch of two without prompt lengths (`lens` defaults to the full cond), seeded inputs; the reference's output is
    kept so the oracle is compared with it wherever the tests run."""
    cfg = tiny_dit()
    sd = O.synthetic_state_dict(cfg, seed=1)
    model = build_reference(cfg, sd)
    g = torch.Generator().manual_seed(0)
    cond = torch.randn(2, 20, 100, generator=g)
    text = torch.randint(0, 50, (2, 25), generator=g)
    dur = torch.tensor([60, 44])
    with torch.no_grad():
        out, _ = model.sample(cond=cond, text=text, duration=dur, steps=3, cfg_strength=2.0, sway_sampling_coef=-1.0,
                              seed=1)
    res = O.sample(sd, cfg, cond, text, dur, steps=3, cfg_strength=2.0, sway_sampling_coef=-1.0, seed=1)
    print("[ref_tiny_b2] oracle-vs-ref rel-L2", rel_l2(res.out, out))
    np.savez_compressed(os.path.join(GOLD, "ref_tiny_b2_nolens.npz"), cond=cond.numpy(), text=text.numpy(),
                        duration=dur.numpy(), out=out.numpy())


def model_configs_golden():
    """The `model` section of the reference's configs/<name>.yaml for every model api.MODEL_ARCH restates."""
    import json

    import yaml

    from f5_tts_b200 import api

    cfg_dir = os.path.join(ref_shims.REFERENCE_SRC, "f5_tts", "configs")
    table = {name: yaml.safe_load(open(os.path.join(cfg_dir, name + ".yaml")))["model"] for name in sorted(api.MODEL_ARCH)}
    with open(os.path.join(GOLD, "model_configs.json"), "w") as f:
        json.dump(table, f, indent=1, sort_keys=True)
        f.write("\n")


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 8)
    mel_golden()
    istft_golden()
    vocos_golden()
    per_op_goldens()
    model_configs_golden()
    ref_tiny_b2_golden()
    # tiny end-to-end cases: every branch of sample()
    run_case("dit_tiny_b1_wave", tiny_dit(), B=1, n_ref=20, nt=24, durations=64, steps=4, cfg_strength=2.0,
             sway=-1.0, seed=3, wave=True)
    run_case("dit_tiny_b3_varlen", tiny_dit(), B=3, n_ref=30, nt=40, durations=[90, 64, 77], lens=[30, 18, 25],
             steps=5, cfg_strength=2.0, sway=-1.0, seed=5, text_pad=[40, 25, 33])
    run_case("dit_tiny_b3_attnmask", tiny_dit(attn_mask_enabled=True), B=3, n_ref=30, nt=40,
             durations=[90, 64, 77], lens=[30, 18, 25], steps=4, cfg_strength=2.0, sway=-1.0, seed=5,
             text_pad=[40, 25, 33])
    run_case("dit_tiny_v1style_b2", tiny_dit(text_mask_padding=True, pe_attn_head=None), B=2, n_ref=24, nt=30,
             durations=[80, 50], lens=[24, 20], steps=6, cfg_strength=2.0, sway=-1.0, seed=6, text_pad=[30, 21])
    run_case("dit_tiny_nocfg_nosway", tiny_dit(), B=1, n_ref=16, nt=90, durations=40, steps=3, cfg_strength=0.0,
             sway=None, seed=8)  # also exercises duration = max(n_text, lens) + 1 (cfm.py:134-137)
    run_case("unett_tiny_b2", tiny_unett(), B=2, n_ref=24, nt=30, durations=[70, 50], lens=[24, 20], steps=4,
             cfg_strength=2.0, sway=-1.0, seed=4, text_pad=[30, 21])
    # full-width cases (weights regenerated from the seed by the tests)
    run_case("f5base_b1_n192", O.f5tts_base(), B=1, n_ref=58, nt=31, durations=192, steps=4, cfg_strength=2.0,
             sway=-1.0, seed=0)
    run_case("f5base_b2_varlen", O.f5tts_base(), B=2, n_ref=50, nt=28, durations=[160, 120], lens=[50, 36], steps=2,
             cfg_strength=2.0, sway=-1.0, seed=1, text_pad=[28, 20])
    run_case("f5v1base_b1_n128", O.f5tts_v1_base(), B=1, n_ref=40, nt=20, durations=128, steps=2, cfg_strength=2.0,
             sway=-1.0, seed=2)
    run_case("e2base_b1_n128", O.e2tts_base(), B=1, n_ref=40, nt=20, durations=128, steps=2, cfg_strength=2.0,
             sway=-1.0, seed=2, wseed=99)


if __name__ == "__main__":
    main()
