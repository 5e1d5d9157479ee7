"""CPU: host logic of the inference-process layer (SURVEY.md §8a rows a19 / a20) — checkpoint loading in the released
layouts, wav reading, and the chunk loop of infer_batch_process (slicing, RMS gain, cross-fade, spectrogram concat)
with the sampler and vocoder replaced by recording fakes.  No kernel is called."""
import os
import wave

import numpy as np
import pytest
import torch

from f5_tts_b200 import infer
from f5_tts_b200.model import CFM, DiT

TINY = dict(dim=128, depth=2, heads=2, ff_mult=2, text_dim=64, conv_layers=1, text_mask_padding=False, pe_attn_head=1)


def _vocab(tmp_path, n=40):
    p = tmp_path / "vocab.txt"
    p.write_text("\n".join([" "] + [chr(ord("a") + i % 26) + ("" if i < 26 else str(i)) for i in range(n - 1)]) + "\n")
    return str(p), n


def _reference_state(model):
    g = torch.Generator().manual_seed(5)
    return {k: torch.randn(v.shape, generator=g) * 0.05 for k, v in model.state_dict().items()}


@pytest.mark.parametrize("fmt", ["safetensors", "pt_ema", "pt_model"])
def test_load_model_and_checkpoint_layouts(tmp_path, fmt):
    """utils_infer.py:190-232: EMA safetensors (`ema_model.` prefix + initted/step), .pt with ema_model_state_dict
    (legacy mel_spec buffers dropped) and .pt with model_state_dict (use_ema=False)."""
    vocab, n = _vocab(tmp_path)
    probe = infer.load_model(DiT, TINY, "", vocab_file=vocab, device="cpu")
    assert isinstance(probe, CFM) and probe.transformer.text_embed.text_embed.weight.shape[0] == n + 1
    want = _reference_state(probe)
    if fmt == "safetensors":
        from safetensors.torch import save_file

        sd = {"ema_model." + k: v for k, v in want.items()}
        sd["initted"], sd["step"] = torch.tensor(True), torch.tensor(7)
        path = str(tmp_path / "model.safetensors")
        save_file(sd, path)
        use_ema = True
    elif fmt == "pt_ema":
        sd = {"ema_model." + k: v for k, v in want.items()}
        sd["initted"], sd["step"] = torch.tensor(True), torch.tensor(7)
        sd["ema_model.mel_spec.mel_stft.mel_scale.fb"] = torch.zeros(3)        # legacy buffers (utils_infer.py:214-219)
        sd["ema_model.mel_spec.mel_stft.spectrogram.window"] = torch.zeros(3)
        path = str(tmp_path / "model.pt")
        torch.save({"ema_model_state_dict": sd}, path)
        use_ema = True
    else:
        path = str(tmp_path / "model.pt")
        torch.save({"model_state_dict": want}, path)
        use_ema = False
    model = infer.load_model(DiT, TINY, path, vocab_file=vocab, use_ema=use_ema, device="cpu")
    got = model.state_dict()
    assert set(got) == set(want)
    for k in want:
        assert torch.equal(got[k].float(), want[k]), k
    assert next(model.parameters()).dtype == torch.float32  # fp16 only on CUDA (utils_infer.py:190-199)


def test_load_model_needs_vocab():
    with pytest.raises(FileNotFoundError):
        infer.load_model(DiT, TINY, "", vocab_file="", device="cpu")


def test_load_wav_pcm16(tmp_path):
    sr, n = 16000, 800
    x = (np.sin(np.arange(n) * 0.05) * 12000).astype("<i2")
    stereo = np.stack([x, -x], axis=1)
    p = str(tmp_path / "a.wav")
    with wave.open(p, "wb") as f:
        f.setnchannels(2)
        f.setsampwidth(2)
        f.setframerate(sr)
        f.writeframes(stereo.tobytes())
    audio, got_sr = infer._load_wav(p)
    assert got_sr == sr and audio.shape == (2, n) and audio.dtype == torch.float32
    assert torch.allclose(audio[0], torch.from_numpy(x.astype(np.float32) / 32768.0))
    assert torch.allclose(audio[1], -audio[0], atol=1 / 32768.0)


class _FakeModel:
    """Records the sampler calls of `_infer_basic` (utils_infer.py:477-520) and returns a ramp mel.  A request with several
    text chunks arrives as ONE batched call (prompt mel expanded over the batch, per-chunk durations, exact_varlen)."""

    def __init__(self):
        self.calls = []

    def mel_spec(self, audio, frames_last=False):  # [1, nw] -> [1, n, 100]; the value marks "computed from the prompt"
        assert not frames_last
        return audio[:, : (audio.shape[-1] // 256) * 256].reshape(1, -1, 256)[:, :, :100].contiguous()

    def sample(self, cond, text, duration, steps, cfg_strength, sway_sampling_coef, lens=None, exact_varlen=False):
        durs = [duration] if isinstance(duration, int) else [int(d) for d in duration]
        self.calls.append(dict(cond=cond.clone(), text=text, duration=durs, steps=steps, cfg=cfg_strength,
                               sway=sway_sampling_coef, lens=lens, exact=exact_varlen))
        mel = torch.arange(max(durs), dtype=torch.float32).view(1, -1, 1).repeat(len(durs), 1, 100)
        return mel, None


class _FakeVocoder:
    def decode(self, mel):  # [1, 100, n] -> [1, 256 (n - 1)], constant 0.5 so gains are visible
        return torch.full((1, 256 * (mel.shape[-1] - 1)), 0.5)


def test_infer_batch_process_chunk_loop():
    sr = infer.target_sample_rate
    ref = torch.full((2, sr), 0.02)  # 1 s stereo, RMS 0.02 < target 0.1 -> gain 5 in, 1/5 out
    ref_text = "hello there."
    batches = ["first chunk of text.", "second one, a bit longer than the first."]
    model, voc = _FakeModel(), _FakeVocoder()
    out = list(infer.infer_batch_process((ref, sr), ref_text, batches, model, voc, nfe_step=7, cfg_strength=1.5,
                                         sway_sampling_coef=-0.5, cross_fade_duration=0.1, device="cpu"))
    assert len(out) == 1
    wave_np, got_sr, spec = out[0]
    assert got_sr == sr
    ref_len = sr // infer.hop_length
    assert len(model.calls) == 1                                           # both chunks in one batched sampler call
    c = model.calls[0]
    assert c["steps"] == 7 and c["cfg"] == 1.5 and c["sway"] == -0.5 and c["exact"] is True
    assert c["cond"].shape == (2, ref_len, 100)                            # prompt mel of the mono mix, once per chunk
    assert torch.allclose(c["cond"], torch.full((2, ref_len, 100), 0.1), atol=1e-6)  # RMS-normalised to 0.1
    assert c["lens"].tolist() == [ref_len, ref_len] and len(c["text"]) == 2
    # duration heuristic: ref frames + ref frames / ref bytes * gen bytes / speed (utils_infer.py:487-493)
    rt = ref_text + " "
    durs = [ref_len + int(ref_len / len(rt.encode()) * len(b.encode()) / 1.0) for b in batches]
    assert c["duration"] == durs
    # per chunk: generated part only, vocoded, gain undone; then cross-faded
    lens = [256 * (d - ref_len - 1) for d in durs]
    fade = int(0.1 * sr)
    assert len(wave_np) == lens[0] + lens[1] - fade
    assert np.allclose(wave_np, 0.5 * 0.02 / 0.1, atol=1e-6)               # constant signal survives the linear fade
    assert spec.shape == (100, (durs[0] - ref_len) + (durs[1] - ref_len))
    assert spec[0, 0] == ref_len and spec[0, durs[0] - ref_len] == ref_len  # each chunk starts right after the prompt


def test_infer_batch_process_streaming_and_short_text():
    sr = infer.target_sample_rate
    ref = torch.full((1, sr), 0.2)  # louder than target: no gain either way
    model, voc = _FakeModel(), _FakeVocoder()
    chunks = list(infer.infer_batch_process((ref, sr), "ok then.", ["hi."], model, voc, device="cpu", streaming=True,
                                            chunk_size=1000))
    ref_len = sr // infer.hop_length
    # < 10 bytes of text -> local speed 0.3 (utils_infer.py:479-481)
    dur = ref_len + int(ref_len / len("ok then. ".encode()) * len("hi.".encode()) / 0.3)
    assert model.calls[0]["duration"] == [dur] and model.calls[0]["cond"].shape == (1, sr)
    total = sum(len(c[0]) for c in chunks)
    assert total == 256 * (dur - ref_len - 1) and all(c[1] == sr for c in chunks)
    assert all(len(c[0]) <= 1000 for c in chunks)
    assert np.allclose(np.concatenate([c[0] for c in chunks]), 0.5)


def test_infer_process_empty_text(tmp_path):
    sr = infer.target_sample_rate
    ref = torch.full((1, 2 * sr), 0.1)
    wav, got_sr, spec = infer.infer_process((ref, sr), "some reference text.", "", _FakeModel(), _FakeVocoder(), device="cpu")
    assert wav is None and spec is None and got_sr == sr


def test_api_model_table_matches_reference_configs(golden_dir):
    """api.MODEL_ARCH restates configs/*.yaml `model.arch` (hydra is not installed here); pinned against the `model`
    sections of the reference's own files (model_configs.json, written by oracle/make_golden.py)."""
    import json

    from f5_tts_b200 import api
    from f5_tts_b200.model import UNetT

    with open(os.path.join(golden_dir, "model_configs.json")) as f:
        ref_configs = json.load(f)
    for name, (cls, arch) in api.MODEL_ARCH.items():
        ref = ref_configs[name]
        assert ref["backbone"] == cls.__name__ and (cls is UNetT) == (ref["backbone"] == "UNetT")
        ref_arch = {k: v for k, v in ref["arch"].items() if k != "checkpoint_activations"}  # training-only switch
        assert {k: arch[k] for k in ref_arch if k in arch} == {k: v for k, v in ref_arch.items() if k in arch}, name
        assert set(arch) <= set(ref_arch), (name, set(arch) - set(ref_arch))
        for k in set(ref_arch) - set(arch):  # anything we leave out must be the reference's inactive default
            assert ref_arch[k] in (None, False, "torch"), (name, k, ref_arch[k])
        assert ref["mel_spec"]["mel_spec_type"] == "vocos" and ref["mel_spec"]["n_mel_channels"] == infer.n_mel_channels
        assert ref["mel_spec"]["hop_length"] == infer.hop_length and ref["mel_spec"]["n_fft"] == infer.n_fft


def test_api_rejects_unknown_model_and_exports_wav(tmp_path):
    from f5_tts_b200 import api

    with pytest.raises(ValueError):
        api.F5TTS(model="nope", ckpt_file="x", vocab_file="y")
    obj = api.F5TTS.__new__(api.F5TTS)  # export helpers do not need a loaded model
    obj.target_sample_rate = 24000
    p = str(tmp_path / "o.wav")
    obj.export_wav(np.array([0.0, 0.5, -2.0], dtype=np.float32), p)
    audio, sr = infer._load_wav(p)
    assert sr == 24000 and torch.allclose(audio[0], torch.tensor([0.0, 0.5, -1.0]), atol=1e-4)


def test_load_vocoder_local_layout(tmp_path):
    """utils_infer.py:118-129: `config.yaml` + `pytorch_model.bin` of charactr/vocos-mel-24khz read from a local folder;
    the state dict (incl. the feature-extractor buffers the checkpoint carries) loads with strict=True."""
    import yaml

    from oracle import f5_oracle as O  # test-only: synthetic weights in the released vocos key layout

    cfg = {
        "feature_extractor": {"class_path": "vocos.feature_extractors.MelSpectrogramFeatures",
                              "init_args": {"sample_rate": 24000, "n_fft": 1024, "hop_length": 256, "n_mels": 100,
                                            "padding": "center"}},
        "backbone": {"class_path": "vocos.models.VocosBackbone",
                     "init_args": {"input_channels": 100, "dim": 512, "intermediate_dim": 1536, "num_layers": 8}},
        "head": {"class_path": "vocos.heads.ISTFTHead",
                 "init_args": {"dim": 512, "n_fft": 1024, "hop_length": 256, "padding": "center"}},
    }
    (tmp_path / "config.yaml").write_text(yaml.safe_dump(cfg))
    sd = O.synthetic_vocos_state_dict()
    # the released checkpoint also carries the (unused at decode time) feature-extractor buffers
    sd["feature_extractor.mel_spec.spectrogram.window"] = torch.hann_window(1024)
    sd["feature_extractor.mel_spec.mel_scale.fb"] = O.mel_filterbank()
    torch.save(sd, str(tmp_path / "pytorch_model.bin"))
    voc = infer.load_vocoder("vocos", is_local=True, local_path=str(tmp_path), device="cpu")
    got = voc.state_dict()
    assert set(got) == set(sd)
    for k, v in sd.items():
        assert torch.equal(got[k], v), k
    assert not voc.training
    with pytest.raises(NotImplementedError):
        infer.load_vocoder("bigvgan", is_local=True, local_path=str(tmp_path), device="cpu")
    with pytest.raises(Exception):  # decode has no CPU path
        voc.decode(torch.zeros(1, 100, 8))


def test_segmentation_without_jieba_follows_jieba_rules():
    """ADVICE r1: the no-rjieba fallback must tokenise like jieba (HMM mode) for non-Chinese text — decimals and
    percentages stay whole, quotes after punctuation get no space (model/utils.py:148-185 downstream of rjieba.cut)."""
    seg = infer._segment_no_chinese
    assert seg("pi is 3.14, v2.10 at 50% off.") == ["pi", " ", "is", " ", "3.14", ",", " ", "v2.10", " ", "at", " ", "50%",
                                                     " ", "off", "."]
    assert seg("hello.'quote' ok") == ["hello", ".", "'", "quote", "'", " ", "ok"]
    assert seg("a-b_c") == ["a", "-", "b", "_", "c"]
    conv = lambda t: "".join(infer.convert_char_to_pinyin([t])[0])  # noqa: E731
    assert conv("pi is 3.14.") == "pi is 3.14."          # not "3. 14"
    assert conv("hello.'quote'") == "hello.'quote'"      # no space between the punctuation and the quote
    assert conv("say:hi") == "say:hi" and conv("ab,cd") == "ab, cd"  # utils.py:172-174: space before a word unless after " :'\""
    try:
        import rjieba  # noqa: F401
    except Exception:  # noqa: BLE001
        with pytest.raises(RuntimeError):
            infer.convert_char_to_pinyin(["你好"])
