"""CPU: pin the oracle restatement (oracle/f5_oracle.py) against vectors produced by the UNMODIFIED
reference (tests/golden/*.npz, written by oracle/make_golden.py).  fp32-vs-fp32 on the same host, so
the bar is tight: rel-L2 <= 1e-5 (observed 0.0 at generation time)."""
import ast
import os

import numpy as np
import pytest
import torch

from oracle import f5_oracle as O

TOL = 1e-5


def _cfg_from_repr(s: str) -> O.ArchConfig:
    body = s[s.index("(") + 1: s.rindex(")")]
    kw = {}
    for part in body.split(", "):
        k, v = part.split("=")
        kw[k] = ast.literal_eval(v)
    return O.ArchConfig(**kw)


def _rel(a, b):
    return float((a - b).norm() / b.norm())


def _run_case(golden_dir, name):
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    cfg = _cfg_from_repr(str(z["cfg"]))
    sd = O.synthetic_state_dict(cfg, seed=int(z["wseed"]))
    dur = z["duration"]
    duration = int(dur) if dur.ndim == 0 else torch.from_numpy(dur).long()
    lens = torch.from_numpy(z["lens"]).long() if z["lens"].size else None
    sway = None if np.isnan(z["sway"]) else float(z["sway"])
    res = O.sample(sd, cfg, torch.from_numpy(z["cond"]), torch.from_numpy(z["text"]), duration, lens=lens,
                   steps=int(z["steps"]), cfg_strength=float(z["cfg_strength"]), sway_sampling_coef=sway,
                   seed=int(z["seed"]))
    assert torch.equal(res.y0, torch.from_numpy(z["y0"])), "noise init must follow cfm.py:196-201 exactly"
    assert _rel(res.trajectory[1], torch.from_numpy(z["traj_1"])) <= TOL
    assert _rel(res.out, torch.from_numpy(z["out"])) <= TOL


@pytest.mark.parametrize("name", ["dit_tiny_b1_wave", "dit_tiny_b3_varlen", "dit_tiny_b3_attnmask",
                                  "dit_tiny_v1style_b2", "dit_tiny_nocfg_nosway", "unett_tiny_b2"])
def test_sample_tiny(golden_dir, name):
    _run_case(golden_dir, name)


@pytest.mark.slow
@pytest.mark.parametrize("name", ["f5base_b1_n192", "f5base_b2_varlen", "f5v1base_b1_n128", "e2base_b1_n128"])
def test_sample_full_width(golden_dir, name):
    _run_case(golden_dir, name)


def test_mel_frontend(golden_dir):
    z = np.load(os.path.join(golden_dir, "mel_vocos.npz"))
    mel = O.mel_spectrogram(torch.from_numpy(z["wav"]))
    assert mel.shape == z["mel"].shape
    assert float((mel - torch.from_numpy(z["mel"])).abs().max()) <= 1e-4


def test_mel_frontend_vs_torchaudio():
    import torchaudio

    wav = 0.1 * torch.randn(1, 5000, generator=torch.Generator().manual_seed(3))
    ta = torchaudio.transforms.MelSpectrogram(sample_rate=24000, n_fft=1024, win_length=1024, hop_length=256,
                                              n_mels=100, power=1, center=True, normalized=False, norm=None)
    ref = ta(wav).clamp(min=1e-5).log()
    assert float((O.mel_spectrogram(wav) - ref).abs().max()) <= 1e-4


def test_istft(golden_dir):
    z = np.load(os.path.join(golden_dir, "istft_torch.npz"))
    spec = torch.complex(torch.from_numpy(z["re"]), torch.from_numpy(z["im"]))
    wav = O.istft_center(spec)
    assert wav.shape[-1] == 256 * (spec.shape[-1] - 1)
    assert float((wav - torch.from_numpy(z["wav"])).abs().max()) <= 1e-5
    live = torch.istft(spec, 1024, 256, 1024, torch.hann_window(1024), center=True)
    assert float((wav - live).abs().max()) <= 1e-5


def test_vocos_frozen(golden_dir):
    z = np.load(os.path.join(golden_dir, "vocos_oracle_frozen.npz"))
    wav = O.vocos_decode(O.synthetic_vocos_state_dict(), torch.from_numpy(z["mel"]))
    assert _rel(wav, torch.from_numpy(z["wav"])) <= 1e-5


def test_per_op(golden_dir):
    z = np.load(os.path.join(golden_dir, "per_op_f5base.npz"))
    cfg = O.f5tts_base()
    sd = O.synthetic_state_dict(cfg, seed=1234)
    x = torch.from_numpy(z["x"])
    B, N, _ = x.shape
    t_emb = O.timestep_embedding(sd, torch.from_numpy(z["t"]))
    assert _rel(t_emb, torch.from_numpy(z["time_embed"])) <= TOL
    ang = O.rope_angles(N)
    assert _rel(ang[None], torch.from_numpy(z["rope_freqs"])) <= TOL
    mask = O.lens_to_mask(torch.tensor([64, 45]))
    assert _rel(O.dit_block(sd, cfg, 3, x, t_emb, None, ang), torch.from_numpy(z["block3_nomask"])) <= TOL
    assert _rel(O.dit_block(sd, cfg, 3, x, t_emb, mask, ang), torch.from_numpy(z["block3_mask"])) <= TOL
    assert _rel(O.conv_position_embedding(sd, x, mask), torch.from_numpy(z["convpos_mask"])) <= TOL
    assert _rel(O.conv_position_embedding(sd, x, None), torch.from_numpy(z["convpos_nomask"])) <= TOL
    text = torch.from_numpy(z["text_in"])
    assert _rel(O.text_embedding_dit(sd, cfg, text, N, False), torch.from_numpy(z["text_embed_cond"])) <= TOL
    assert _rel(O.text_embedding_dit(sd, cfg, text, N, True), torch.from_numpy(z["text_embed_uncond"])) <= TOL
    assert _rel(O.text_embedding_dit(sd, cfg, text, mask.sum(1), False),
                torch.from_numpy(z["text_embed_cond_varlen"])) <= TOL


def test_time_grid():
    t = O.time_grid(16, -1.0)
    assert t.shape[0] == 17
    raw = torch.tensor(O.EPSS[16]) / 32.0
    assert torch.allclose(t, 1 - torch.cos(torch.pi / 2 * raw), atol=1e-6)
    assert torch.allclose(O.time_grid(32, None), torch.linspace(0, 1, 33))


def test_live_reference_if_present(golden_dir):
    """A batch of two without `lens` against the reference's output on the same inputs (ref_tiny_b2_nolens.npz, written
    by oracle/make_golden.py from the unmodified reference)."""
    from oracle import make_golden as MG

    z = np.load(os.path.join(golden_dir, "ref_tiny_b2_nolens.npz"))
    cfg = MG.tiny_dit()
    sd = O.synthetic_state_dict(cfg, seed=1)
    res = O.sample(sd, cfg, torch.from_numpy(z["cond"]), torch.from_numpy(z["text"]), torch.from_numpy(z["duration"]),
                   steps=3, cfg_strength=2.0, sway_sampling_coef=-1.0, seed=1)
    assert _rel(res.out, torch.from_numpy(z["out"])) <= TOL
