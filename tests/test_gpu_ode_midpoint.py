"""GPU: the midpoint ODE solver (CFM(odeint_kwargs=dict(method="midpoint")), F5TTS(ode_method="midpoint")).

torchdiffeq's fixed-grid midpoint on the caller's grid t[0..S] (cfm.py:218): per step k, with dt = t[k+1] - t[k],
    y_mid = y + f(t[k], y) * dt/2;   y <- y + dt * f(t[k] + dt/2, y_mid)     (trajectory keeps the S + 1 grid points)
The engine runs it as 2S backbone evaluations; the fused CFG + update kernel reads {coef, commit} per evaluation.

  * the reference through the restated solver (tests/golden/*_midpoint.npz, oracle/make_golden_midpoint.py) and the
    CPU oracle on fresh inputs (masked / attn-mask / no-CFG / exact_varlen), rel-L2 <= 5e-3 as in test_gpu_sample.py;
  * the stage structure of one grid step, against torch arithmetic on the engine's own v_out and against two chained
    Euler calls (both bit-exact);
  * graph replay == eager and run-to-run bit-identity with Euler and midpoint calls sharing one workspace;
  * rejection of an unknown f5_sample_args.ode_method; F5TTS(ode_method="midpoint").infer end to end;
  * the full-size cfg2 (EPSS-16) and cfg3-masked shapes against fixtures of the CPU oracle (fullsize marker).
"""
import ast
import ctypes as C
import os

import numpy as np
import pytest
import torch
import yaml

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import f5_tts_b200 as F5  # noqa: E402
import synthdata as SD  # noqa: E402
from f5_tts_b200 import _lib, api, infer  # noqa: E402
from oracle import f5_oracle as O  # noqa: E402
from oracle import ode_midpoint as M  # noqa: E402

DEV = "cuda:0"
TOL = 5e-3
_models = {}


def cfg_from_repr(s: str) -> O.ArchConfig:
    body = s[s.index("(") + 1: s.rindex(")")]
    return O.ArchConfig(**{k: ast.literal_eval(v) for k, v in (p.split("=") for p in body.split(", "))})


def build(cfg, wseed=1234, method="midpoint"):
    """(CFM with `method`, state dict); one backbone resident at a time, shared by both solvers."""
    key = (repr(cfg), wseed)
    if key not in _models:
        _models.clear()
        cls = F5.DiT if cfg.backbone == "DiT" else F5.UNetT
        tr = cls(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, dim_head=cfg.dim_head, ff_mult=cfg.ff_mult,
                 mel_dim=cfg.mel_dim, text_num_embeds=cfg.text_num_embeds, text_dim=cfg.text_dim,
                 text_mask_padding=cfg.text_mask_padding, conv_layers=cfg.conv_layers, pe_attn_head=cfg.pe_attn_head,
                 attn_mask_enabled=cfg.attn_mask_enabled)
        sd = O.synthetic_state_dict(cfg, seed=wseed)
        m = F5.CFM(transformer=tr)
        m.load_state_dict(sd, strict=True)
        _models[key] = (m.to(DEV).transformer, sd)
    tr, sd = _models[key]
    return F5.CFM(transformer=tr, odeint_kwargs=dict(method=method)).to(DEV), sd


def rel(a, b):
    a, b = torch.as_tensor(a).float().cpu(), torch.as_tensor(b).float().cpu()
    return float((a - b).norm() / b.norm())


# ---------------------------------------------------------------------------------------------------------------------
# parity
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["f5base_b1_n192_midpoint", "f5v1base_b1_n128_midpoint", "e2base_b1_n128_midpoint"])
def test_midpoint_vs_reference_golden(golden_dir, name):
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    assert str(z["method"]) == "midpoint"
    model, _ = build(cfg_from_repr(str(z["cfg"])), int(z["wseed"]))
    steps = int(z["steps"])
    out, traj = model.sample(cond=torch.from_numpy(z["cond"]).to(DEV), text=torch.from_numpy(z["text"]).to(DEV),
                             duration=int(z["duration"]), steps=steps, cfg_strength=float(z["cfg_strength"]),
                             sway_sampling_coef=float(z["sway"]), seed=int(z["seed"]),
                             y0=torch.from_numpy(z["y0"]).to(DEV))
    r1, rN = rel(traj[1], z["traj_1"]), rel(out, z["out"])
    print(f"[{name}] step-1 rel-L2 {r1:.3e}  final rel-L2 {rN:.3e}")
    assert traj.shape[0] == steps + 1 and out.shape == z["out"].shape
    assert r1 <= TOL and rN <= TOL


@pytest.mark.parametrize("variant", ["mask_faithful", "attn_mask", "no_cfg"])
def test_midpoint_vs_oracle(variant):
    cfg = O.f5tts_base()
    cfg.attn_mask_enabled = variant == "attn_mask"
    model, sd = build(cfg)
    g = torch.Generator().manual_seed(42)
    kw = dict(steps=2, cfg_strength=2.0, sway_sampling_coef=-1.0, seed=7)
    if variant == "no_cfg":
        args = (torch.randn(1, 30, 100, generator=g), torch.randint(0, 2545, (1, 25), generator=g), 130)
        kw.update(cfg_strength=0.0, sway_sampling_coef=None, steps=3)
    else:
        cond = torch.randn(3, 40, 100, generator=g)
        text = torch.randint(0, 2545, (3, 30), generator=g)
        text[1, 20:] = -1
        args = (cond, text, torch.tensor([150, 97, 131]))
        kw["lens"] = torch.tensor([40, 25, 33])
    ref = M.sample(sd, cfg, *args, **kw, method="midpoint")
    dargs = tuple(a.to(DEV) if torch.is_tensor(a) else a for a in args)
    dkw = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in kw.items()}
    out, traj = model.sample(*dargs, **dkw, y0=ref.y0.to(DEV))
    assert traj.shape[0] == kw["steps"] + 1
    if variant == "attn_mask":  # rows past a sample's duration are not computed in key-masked mode: valid rows only
        durs = args[2].tolist()
        r = rel(torch.cat([out[b, :d].cpu() for b, d in enumerate(durs)]),
                torch.cat([ref.out[b, :d] for b, d in enumerate(durs)]))
        r1 = rel(torch.cat([traj[1][b, :d].cpu() for b, d in enumerate(durs)]),
                 torch.cat([ref.trajectory[1][b, :d] for b, d in enumerate(durs)]))
    else:
        r, r1 = rel(out, ref.out), rel(traj[1], ref.trajectory[1])
    print(f"[midpoint oracle:{variant}] final rel-L2 {r:.3e}  step-1 {r1:.3e}")
    assert r <= TOL and r1 <= TOL


def test_midpoint_exact_varlen_batch_equals_single_calls():
    """infer_batch_process's batched chunk path (exact_varlen) with midpoint == a loop of B = 1 midpoint calls."""
    model, _ = build(O.f5tts_base())
    g = torch.Generator().manual_seed(33)
    n_ref, durs = 60, [420, 150, 297]
    cond = torch.randn(1, n_ref, 100, generator=g)
    text = torch.randint(0, 2545, (3, 50), generator=g)
    text[1, 30:] = -1
    y0 = [torch.randn(1, d, 100, generator=g) for d in durs]
    kw = dict(steps=2, cfg_strength=2.0, sway_sampling_coef=-1.0)
    singles = []
    for b, d in enumerate(durs):
        tb = text[b: b + 1, : int((text[b] != -1).sum())]
        singles.append(model.sample(cond.to(DEV), tb.to(DEV), d, **kw, y0=y0[b].to(DEV))[0])
    y0b = torch.zeros(3, max(durs), 100)
    for b, d in enumerate(durs):
        y0b[b, :d] = y0[b][0]
    out, traj = model.sample(cond.expand(3, -1, -1).contiguous().to(DEV), text.to(DEV), torch.tensor(durs).to(DEV),
                             lens=torch.full((3,), n_ref).to(DEV), **kw, y0=y0b.to(DEV), exact_varlen=True)
    assert traj.shape[0] == 3
    for b, d in enumerate(durs):
        r = rel(out[b, :d], singles[b][0])
        print(f"[midpoint exact_varlen] sample {b} ({d} frames): batched vs single rel-L2 {r:.3e}")
        assert r <= 1e-3


# ---------------------------------------------------------------------------------------------------------------------
# stage structure of one grid step
# ---------------------------------------------------------------------------------------------------------------------
def _engine_call(tr, y0, sc, text, grid, cfg, method):
    """one f5_sample call through the backbone's run(): (trajectory [S+1, B, N, mel], v_out [Be, N, mel])"""
    B, N, mel = y0.shape
    y = y0.clone()
    traj = torch.empty((len(grid), B, N, mel), device=DEV)
    v = torch.empty((2 * B if cfg > 0 else B, N, mel), device=DEV)
    tr.run(y, sc, text, grid, None, cfg, trajectory=traj, v_out=v, ode_method=method)
    torch.cuda.synchronize()
    assert torch.equal(traj[-1], y)
    return traj, v


def test_midpoint_stage_structure():
    """Grid [t0, t1] = [0.25, 0.75]: t0 + dt/2 = 0.5 and dt/2 = 0.25 are exact in fp32, so the half step can be
    replayed as an Euler call on [0.25, 0.5].
      (1) trajectory[1] == y0 + dt * (pr + (pr - nu) * cfg) with pr / nu the v_out of the midpoint evaluation:
          the commit uses the step's base state y0, the full dt and the mid-point velocity;
      (2) v_out == the v_out of an Euler call on [t0 + dt/2, t1] started from the trajectory[1] of an Euler call on
          [t0, t0 + dt/2]: the half step feeds y0 + dt/2 * f(t0, y0) at time t0 + dt/2 to the second evaluation."""
    model, _ = build(O.f5tts_base())
    tr = model.transformer
    g = torch.Generator().manual_seed(5)
    B, N, cfg = 1, 150, 2.0
    sc = torch.zeros(B, N, 100)
    sc[:, :40] = torch.randn(B, 40, 100, generator=g)
    sc, text = sc.to(DEV), torch.randint(0, 2545, (B, 40), generator=g).to(DEV)
    y0 = torch.randn(B, N, 100, generator=g).to(DEV)
    t0, t1 = 0.25, 0.75
    dt = t1 - t0
    traj, v = _engine_call(tr, y0, sc, text, [t0, t1], cfg, "midpoint")
    assert torch.equal(traj[0], y0)
    pr, nu = v[:B], v[B:]
    want = y0 + dt * (pr + (pr - nu) * cfg)
    print(f"[stage] commit vs y0 + dt * g(v_out): rel-L2 {rel(traj[1], want):.3e}")
    assert torch.equal(traj[1], want)
    tr_a, _ = _engine_call(tr, y0, sc, text, [t0, t0 + dt / 2], cfg, "euler")
    _, v_b = _engine_call(tr, tr_a[1].contiguous(), sc, text, [t0 + dt / 2, t1], cfg, "euler")
    print(f"[stage] mid-point v_out vs chained Euler calls: rel-L2 {rel(v, v_b):.3e}")
    assert torch.equal(v, v_b)


# ---------------------------------------------------------------------------------------------------------------------
# graph cache, determinism, rejection
# ---------------------------------------------------------------------------------------------------------------------
def test_graph_equals_eager_with_euler_and_midpoint_sharing_a_workspace():
    """An Euler call with 2S steps and a midpoint call with S steps run the same number of evaluations on the same
    workspace, so they replay one captured graph; the per-call OdeStage table keeps them apart."""
    mid, _ = build(O.f5tts_base())
    eul = F5.CFM(transformer=mid.transformer).to(DEV)
    g = torch.Generator().manual_seed(1)
    cond = torch.randn(1, 50, 100, generator=g).to(DEV)
    text = torch.randint(0, 2545, (1, 40), generator=g).to(DEV)
    kw = dict(cfg_strength=2.0, sway_sampling_coef=-1.0, seed=3, use_epss=False)
    runs = {"euler": [], "midpoint": []}
    for graph in (True, True, False):
        for name, m, steps in (("euler", eul, 6), ("midpoint", mid, 3)):
            m.use_cuda_graph = graph
            out, traj = m.sample(cond, text, 200, steps=steps, **kw)
            runs[name].append((out, traj))
    for name, rs in runs.items():
        (a, ta), (b, tb), (c, tc) = rs
        assert torch.equal(a, b) and torch.equal(ta, tb), f"{name}: run to run"
        assert torch.equal(a, c) and torch.equal(ta, tc), f"{name}: graph replay vs eager"
    assert runs["euler"][0][1].shape[0] == 7 and runs["midpoint"][0][1].shape[0] == 4
    # the two solvers share grid points t = 0, 1/3, 2/3, 1 (linspace 6 and 3 + the same sway) yet differ there
    assert rel(runs["euler"][0][0], runs["midpoint"][0][0]) > 1e-4


def test_unknown_ode_method_is_rejected():
    model, _ = build(O.f5tts_base())
    tr = model.transformer
    L = _lib.lib()
    ws = torch.empty(1 << 16, dtype=torch.uint8, device=DEV)
    for bad in (2, -1):
        a = _lib.SampleArgs()
        a.B, a.N, a.nt, a.steps = 1, 16, 4, 1
        a.ode_method = bad
        rc = L.f5_sample(tr.engine()["handle"], C.byref(a), ws.data_ptr(), ws.numel(),
                         torch.cuda.current_stream().cuda_stream)
        msg = L.f5_last_error().decode()
        assert rc != 0 and "ode_method" in msg, (rc, msg)
    with pytest.raises(NotImplementedError):
        tr.run(torch.zeros(1, 16, 100, device=DEV), torch.zeros(1, 16, 100, device=DEV),
               torch.zeros(1, 4, dtype=torch.int64, device=DEV), [0.0, 1.0], None, 2.0, ode_method="rk4")


# ---------------------------------------------------------------------------------------------------------------------
# top level: F5TTS(ode_method="midpoint").infer
# ---------------------------------------------------------------------------------------------------------------------
REF_TEXT = "Some call me nature, others call me mother nature."  # infer/examples/basic/basic.toml
GEN_SHORT = "I don't really care what you call me."


def test_f5tts_infer_midpoint(tmp_path, golden_dir):
    from safetensors.torch import save_file

    sd = SD.synthetic_state_dict(SD.f5tts_base(), seed=1234)
    ema = {"ema_model." + k: v for k, v in sd.items()}
    ema["initted"], ema["step"] = torch.tensor(True), torch.tensor(1)
    ckpt = str(tmp_path / "model_1.safetensors")
    save_file(ema, ckpt)
    vdir = tmp_path / "vocos"
    vdir.mkdir()
    (vdir / "config.yaml").write_text(yaml.safe_dump(
        {"feature_extractor": {"class_path": "vocos.feature_extractors.MelSpectrogramFeatures",
                               "init_args": {"sample_rate": 24000, "n_fft": 1024, "hop_length": 256, "n_mels": 100,
                                             "padding": "center"}},
         "backbone": {"class_path": "vocos.models.VocosBackbone",
                      "init_args": {"input_channels": 100, "dim": 512, "intermediate_dim": 1536, "num_layers": 8}},
         "head": {"class_path": "vocos.heads.ISTFTHead",
                  "init_args": {"dim": 512, "n_fft": 1024, "hop_length": 256, "padding": "center"}}}))
    full = dict(SD.synthetic_vocos_state_dict())
    full["feature_extractor.mel_spec.spectrogram.window"] = torch.hann_window(1024)
    full["feature_extractor.mel_spec.mel_scale.fb"] = O.mel_filterbank()
    torch.save(full, str(vdir / "pytorch_model.bin"))
    ref = os.path.join(golden_dir, "basic_ref_en.wav")
    tts = api.F5TTS(model="F5TTS_Base", ckpt_file=ckpt, vocab_file=os.path.join(golden_dir, "vocab.txt"),
                    ode_method="midpoint", vocoder_local_path=str(vdir), device=DEV)
    assert tts.ema_model.odeint_kwargs["method"] == "midpoint"
    nfe, seed = 4, 1234
    wav, sr, spec = tts.infer(ref, REF_TEXT, GEN_SHORT, nfe_step=nfe, seed=seed, show_info=lambda *_: None)
    ref_len = 127987 // 256
    ref_text = REF_TEXT + "  "  # preprocess_ref_audio_text and infer_batch_process each append a space
    duration = ref_len + int(ref_len / len(ref_text.encode()) * len(GEN_SHORT.encode()))
    assert sr == 24000 and spec.shape == (100, duration - ref_len) and wav.shape == (256 * (duration - ref_len - 1),)
    assert np.isfinite(wav).all() and float(np.abs(wav).max()) > 0
    # the same sampler call made directly: same prompt wave, tokens, duration and seeded device noise
    audio, _ = infer._load_wav(ref)
    rms = torch.sqrt(torch.mean(torch.square(audio)))
    if rms < 0.1:
        audio = audio * 0.1 / rms
    tokens = infer.convert_char_to_pinyin([ref_text + GEN_SHORT])
    api.seed_everything(seed)
    with torch.inference_mode():
        out, traj = tts.ema_model.sample(cond=audio.to(DEV), text=tokens, duration=duration, steps=nfe, cfg_strength=2,
                                         sway_sampling_coef=-1)
    assert traj.shape[0] == nfe + 1
    mel = out[0, ref_len:, :].to(torch.float32).T.cpu().numpy()
    assert np.array_equal(spec, mel)


# ---------------------------------------------------------------------------------------------------------------------
# full size
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.fullsize
@pytest.mark.parametrize("name", ["cfg2_midpoint16", "cfg3_masked_midpoint4"])
def test_fullsize_midpoint(golden_dir, name):
    """cfg2 (B=1, 938 frames, EPSS-16 grid: 32 evaluations, the cost of Euler NFE 32) and cfg3 masked (B=8, 469..1875
    frames, 4 steps) against tests/golden/fullsize_<name>.npz (oracle/make_golden_midpoint.py): every `stride`-th
    generated row of every utterance (3 for cfg2, 12 for cfg3) after step 1 and at the end."""
    from oracle.make_golden_fullsize import draw_y0

    z = np.load(os.path.join(golden_dir, f"fullsize_{name}.npz"))
    assert str(z["method"]) == "midpoint"
    cfg = getattr(SD, str(z["arch"]))()
    cfg.attn_mask_enabled = bool(z["attn_mask_enabled"])
    w, steps, stride = SD.WORKLOADS[str(z["workload"])], int(z["steps"]), int(z["stride"])
    model, _ = build(cfg, int(z["wseed"]))
    wav, text, duration, lens = SD.synth_inputs(w)
    cond = O.mel_spectrogram(wav).permute(0, 2, 1).contiguous()
    y0 = draw_y0(duration, cfg.mel_dim, seed=int(z["seed"]))
    chk = np.array([float(y0.double().sum()), float(y0.double().abs().sum())])
    assert np.allclose(chk, z["y0_checksum"], rtol=1e-12), "the CPU generator drew different noise than the fixture's"
    out, traj = model.sample(cond.to(DEV), text.to(DEV), duration.to(DEV), lens=lens.to(DEV), steps=steps,
                             cfg_strength=SD.CFG_STRENGTH, sway_sampling_coef=SD.SWAY, seed=int(z["seed"]),
                             y0=y0.to(DEV))
    assert traj.shape[0] == steps + 1
    g1, gN = torch.from_numpy(z["step1"]), torch.from_numpy(z["final"])
    worst, at = 0.0, 0
    for b in range(w["B"]):
        sl = slice(int(lens[b]), int(duration[b]), stride)
        n = len(range(*sl.indices(int(duration[b]))))
        r1, rN = rel(traj[1][b, sl], g1[at: at + n]), rel(out[b, sl], gN[at: at + n])
        at += n
        worst = max(worst, r1, rN)
        print(f"[{name}] utt {b} frames {int(duration[b])}: step-1 {r1:.3e}  final({steps} steps) {rN:.3e}")
    assert at == g1.shape[0] == gN.shape[0]
    assert worst <= TOL
