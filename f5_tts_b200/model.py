"""Host-side mirror of the reference's model surface for the ODE-sampling path.

Same names, constructor arguments, ``state_dict`` keys and call semantics as the reference
(``f5_tts.model.{CFM, DiT, UNetT}``, ``f5_tts.model.modules.MelSpec``), but the modules are only parameter
containers + tensor plumbing: every arithmetic step runs in the hand-written sm_100a kernels of
libf5tts_b200.so.  There is no PyTorch compute fallback — without the library (or off a B200) calls raise.

Reference anchors (relative to /root/reference/src/f5_tts):
  CFM.sample            model/cfm.py:83-229
  DiT                   model/backbones/dit.py:170-370      (forward 319-370)
  UNetT                 model/backbones/unett.py:108-307    (forward 244-307)
  MelSpec               model/modules.py:112-151
  lens_to_mask etc.     model/utils.py:53-58, 88-106, 205-218
"""
from __future__ import annotations

import ctypes as C
import math
import threading
from typing import Callable, Optional

import torch
import torch.nn.functional as F
from torch import nn
from torch.nn.utils.rnn import pad_sequence

from . import _lib

# ----------------------------------------------------------------------------------------------------------------
# small host helpers (model/utils.py)
# ----------------------------------------------------------------------------------------------------------------


def exists(v):
    return v is not None


def default(v, d):
    return v if exists(v) else d


def lens_to_mask(t: torch.Tensor, length: Optional[int] = None) -> torch.Tensor:
    """bool[b, n] with n = max(t) unless given (model/utils.py:53-58)"""
    if length is None:
        length = int(t.amax())
    return torch.arange(length, device=t.device)[None, :] < t[:, None]


def list_str_to_tensor(text: list[str], padding_value=-1) -> torch.Tensor:
    """utf-8 byte tokenizer (model/utils.py:88-91)"""
    rows = [torch.tensor(list(bytes(t, "UTF-8"))) for t in text]
    return pad_sequence(rows, padding_value=padding_value, batch_first=True)


def list_str_to_idx(text, vocab_char_map: dict, padding_value=-1) -> torch.Tensor:
    """char / pinyin-token tokenizer; unknown -> 0 (model/utils.py:99-106)"""
    rows = [torch.tensor([vocab_char_map.get(c, 0) for c in t]) for t in text]
    return pad_sequence(rows, padding_value=padding_value, batch_first=True)


_EPSS = {  # model/utils.py:205-218
    5: [0, 2, 4, 8, 16, 32],
    6: [0, 2, 4, 6, 8, 16, 32],
    7: [0, 2, 4, 6, 8, 16, 24, 32],
    10: [0, 2, 4, 6, 8, 12, 16, 20, 24, 28, 32],
    12: [0, 2, 4, 6, 8, 10, 12, 14, 16, 20, 24, 28, 32],
    16: [0, 1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 14, 16, 20, 24, 28, 32],
}


def get_epss_timesteps(n, device, dtype):
    t = _EPSS.get(n)
    if not t:
        return torch.linspace(0, 1, n + 1, device=device, dtype=dtype)
    return (1 / 32) * torch.tensor(t, device=device, dtype=dtype)


# ----------------------------------------------------------------------------------------------------------------
# parameter trees with the released checkpoint key layout (SURVEY.md §8b)
# ----------------------------------------------------------------------------------------------------------------


def _attach(root: nn.Module, dotted: str, tensor: torch.Tensor, buffer=False):
    *path, leaf = dotted.split(".")
    mod = root
    for name in path:
        if name not in mod._modules:
            mod.add_module(name, nn.Module())
        mod = mod._modules[name]
    if buffer:
        mod.register_buffer(leaf, tensor, persistent=True)
    else:
        mod.register_parameter(leaf, nn.Parameter(tensor, requires_grad=False))


def _backbone_spec(kind: str, *, dim, depth, heads, dim_head, ff_mult, mel_dim, text_num_embeds, text_dim,
                   conv_layers):
    """(key, shape, init) for every tensor of the backbone; identical names to dit.py / unett.py modules."""
    D, T, Mel = dim, text_dim, mel_dim
    inner, ff = heads * dim_head, int(dim * ff_mult)
    out = []

    def lin(p, o, i, bias=True, init="w"):
        out.append((p + ".weight", (o, i), init))
        if bias:
            out.append((p + ".bias", (o,), "zero"))

    lin("time_embed.time_mlp.0", D, 256)
    lin("time_embed.time_mlp.2", D, D)
    out.append(("text_embed.text_embed.weight", (text_num_embeds + 1, T), "w"))
    for i in range(conv_layers):
        b = f"text_embed.text_blocks.{i}."
        out += [(b + "dwconv.weight", (T, 1, 7), "w"), (b + "dwconv.bias", (T,), "zero"),
                (b + "norm.weight", (T,), "one"), (b + "norm.bias", (T,), "zero")]
        lin(b + "pwconv1", 2 * T, T)
        out += [(b + "grn.gamma", (1, 1, 2 * T), "zero"), (b + "grn.beta", (1, 1, 2 * T), "zero")]
        lin(b + "pwconv2", T, 2 * T)
    lin("input_embed.proj", D, 2 * Mel + T)
    for i in (0, 2):
        out += [(f"input_embed.conv_pos_embed.conv1d.{i}.weight", (D, D // 16, 31), "w"),
                (f"input_embed.conv_pos_embed.conv1d.{i}.bias", (D,), "zero")]
    if kind == "DiT":
        for i in range(depth):
            b = f"transformer_blocks.{i}."
            lin(b + "attn_norm.linear", 6 * D, D, init="zero")  # AdaLN-Zero (dit.py:264-274)
            for nm in ("to_q", "to_k", "to_v"):
                lin(b + "attn." + nm, inner, D)
            lin(b + "attn.to_out.0", D, inner)
            lin(b + "ff.ff.0.0", ff, D)
            lin(b + "ff.ff.2", D, ff)
        lin("norm_out.linear", 2 * D, D, init="zero")
        lin("proj_out", Mel, D, init="zero")
    else:
        for i in range(depth):
            b = f"layers.{i}."
            if i >= depth // 2:
                lin(b + "0", D, 2 * D, bias=False)
            out.append((b + "1.g", (D,), "one"))
            for nm in ("to_q", "to_k", "to_v"):
                lin(b + "2." + nm, inner, D)
            lin(b + "2.to_out.0", D, inner)
            out.append((b + "3.g", (D,), "one"))
            lin(b + "4.ff.0.0", ff, D)
            lin(b + "4.ff.2", D, ff)
        out.append(("norm_out.g", (D,), "one"))
        lin("proj_out", Mel, D)
    return out


def _init_tensor(shape, how):
    if how == "zero":
        return torch.zeros(shape)
    if how == "one":
        return torch.ones(shape)
    fan_in = shape[-1] if len(shape) == 2 else int(torch.tensor(shape[1:]).prod())
    return torch.randn(shape) / math.sqrt(max(fan_in, 1))


def _ode_method_id(method: str) -> int:
    """torchdiffeq method name -> f5_sample_args.ode_method; the engine builds the fixed-grid "euler" and "midpoint"."""
    if method not in _lib.ODE_METHODS:
        raise NotImplementedError(f"ODE method {method!r} is not built: the engine implements 'euler' (the shipped "
                                  "default) and 'midpoint'")
    return _lib.ODE_METHODS[method]


def _ode_evals(steps: int, method_id: int) -> int:
    """backbone evaluations of `steps` grid steps: the `evals` argument of f5_sample_workspace_bytes / f5_sample_flops"""
    return 2 * steps if method_id == _lib.ODE_MIDPOINT else steps


class _Backbone(nn.Module):
    """Shared implementation of the `transformer(...)` operator seam (SURVEY.md §8b)."""

    KIND = "DiT"

    def __init__(self, *, dim, depth=8, heads=8, dim_head=64, dropout=0.1, ff_mult=4, mel_dim=100,
                 text_num_embeds=256, text_dim=None, text_mask_padding=True, qk_norm=None, conv_layers=0,
                 pe_attn_head=None, attn_backend="torch", attn_mask_enabled=False, **unsupported):
        super().__init__()
        if qk_norm is not None:
            raise NotImplementedError("qk_norm is null in every shipped config (configs/*.yaml); not built")
        for k in ("text_embedding_average_upsampling", "long_skip_connection", "checkpoint_activations"):
            if unsupported.pop(k, False):
                raise NotImplementedError(f"{k} is off in every shipped config; not built")
        skip = unsupported.pop("skip_connect_type", "concat")
        if skip != "concat":
            raise NotImplementedError("UNetT skip_connect_type other than 'concat' is not built")
        if unsupported:
            raise TypeError(f"unexpected arguments: {sorted(unsupported)}")
        if dim_head != 64:
            raise NotImplementedError("the attention kernel is built for dim_head == 64")
        if text_dim is None:
            text_dim = mel_dim
        self.dim, self.depth, self.heads, self.dim_head = dim, depth, heads, dim_head
        self.ff_inner = int(dim * ff_mult)
        self.mel_dim, self.text_dim, self.text_num_embeds = mel_dim, text_dim, text_num_embeds
        self.text_mask_padding, self.conv_layers = bool(text_mask_padding), conv_layers
        self.pe_attn_head, self.attn_mask_enabled = pe_attn_head, bool(attn_mask_enabled)
        self.attn_backend = attn_backend  # accepted for config compatibility; the B200 kernel is always used
        for key, shape, how in _backbone_spec(self.KIND, dim=dim, depth=depth, heads=heads, dim_head=dim_head,
                                              ff_mult=ff_mult, mel_dim=mel_dim, text_num_embeds=text_num_embeds,
                                              text_dim=text_dim, conv_layers=conv_layers):
            _attach(self, key, _init_tensor(shape, how))
        inv_freq = 1.0 / (10000 ** (torch.arange(0, dim_head, 2).float() / dim_head))
        _attach(self, "rotary_embed.inv_freq", inv_freq, buffer=True)
        self._engine_lock = threading.Lock()
        self._engine_state = None
        self._ws_lock = threading.Lock()
        self._ws_free: dict = {}  # (device, stream) -> [uint8 tensors] not in use by a sample() call

    # -- engine management ------------------------------------------------------------------------------------
    def _fingerprint(self):
        """(address, version, dtype) of every parameter: changes when weights are loaded, moved or edited in place.
        Runs on every engine call, so it walks a cached list of the parameter-holding modules (the module tree is fixed
        after __init__) instead of nn.Module.parameters(), whose recursive generator costs ~1.6 ms for this tree."""
        mods = self.__dict__.get("_param_modules")
        if mods is None:
            mods = [m for m in self.modules() if m._parameters]
            self.__dict__["_param_modules"] = mods
        return tuple((p.data_ptr(), p._version, p.dtype) for m in mods for p in m._parameters.values() if p is not None)

    def engine(self):
        """(handle, keepalive) — re-packs weights to the kernels' layouts when parameters changed."""
        fp = self._fingerprint()
        with self._engine_lock:
            st = self._engine_state
            if st is None or st["fp"] != fp:
                if st is not None:
                    _lib.lib().f5_engine_destroy(st["handle"])
                from .weights import pack_backbone

                st = pack_backbone(self)
                st["fp"] = fp
                self._engine_state = st
            return st

    def __del__(self):
        st = getattr(self, "_engine_state", None)
        if st is not None:
            try:
                _lib.lib().f5_engine_destroy(st["handle"])
            except Exception:
                pass

    def clear_cache(self):
        """Text embeddings are recomputed inside every engine call; nothing is cached across calls."""
        return None

    def _ws_acquire(self, nbytes: int, device, stream: int) -> torch.Tensor:
        """Scratch for one engine call, from a pool keyed on (device, stream).  Concurrent sample() calls (the reference
        samples from a ThreadPoolExecutor, utils_infer.py:540-541) each hold their own buffer; a finished call returns
        it, so the next call — from any thread — reuses the same address and hits the engine's CUDA-graph cache (the
        graph is keyed on the workspace address).  Reuse is stream-ordered, hence the stream in the key."""
        key = (torch.device(device), int(stream))
        with self._ws_lock:
            free = self._ws_free.setdefault(key, [])
            for i, ws in enumerate(free):
                if ws.numel() >= nbytes:
                    return free.pop(i)
            free.clear()  # too small for the current shapes: let them go
        return torch.empty(int(nbytes * 1.05) + 4096, dtype=torch.uint8, device=device)

    def _ws_release(self, ws: torch.Tensor, device, stream: int) -> None:
        with self._ws_lock:
            self._ws_free.setdefault((torch.device(device), int(stream)), []).append(ws)

    def run(self, y, step_cond, text, t_grid, duration, cfg_strength, trajectory=None, v_out=None, use_graph=True,
            exact_varlen=False, ode_method="euler"):
        """One engine call = len(t_grid)-1 steps of the fixed-grid ODE solver `ode_method` ("euler": one backbone
        evaluation per step, "midpoint": two).  All tensors on the CUDA device, fp32 / int64 / int32."""
        st = self.engine()
        L = _lib.lib()
        B, N, mel = y.shape
        steps = len(t_grid) - 1
        assert y.is_contiguous() and step_cond.is_contiguous() and text.is_contiguous()
        assert y.dtype == torch.float32 and step_cond.dtype == torch.float32 and text.dtype == torch.int64
        method = _ode_method_id(ode_method)
        need = L.f5_sample_workspace_bytes(st["handle"], B, N, _ode_evals(steps, method), float(cfg_strength))
        stream = torch.cuda.current_stream(y.device).cuda_stream
        ws = self._ws_acquire(need, y.device, stream)
        tg = (C.c_float * (steps + 1))(*[float(v) for v in t_grid])
        a = _lib.SampleArgs()
        a.B, a.N, a.nt, a.steps = B, N, text.shape[1], steps
        a.text, a.step_cond, a.y = text.data_ptr(), step_cond.data_ptr(), y.data_ptr()
        a.duration = duration.data_ptr() if duration is not None else None
        a.t = tg
        a.cfg_strength = float(cfg_strength)
        a.trajectory = trajectory.data_ptr() if trajectory is not None else None
        a.use_graph = 1 if use_graph else 0
        a.v_out = v_out.data_ptr() if v_out is not None else None
        a.exact_varlen = 1 if (exact_varlen and duration is not None) else 0
        a.ode_method = method
        try:
            with torch.cuda.device(y.device):
                _lib.check(L.f5_sample(st["handle"], C.byref(a), ws.data_ptr(), ws.numel(), stream), "f5_sample")
        finally:
            self._ws_release(ws, y.device, stream)

    def sample_flops(self, B, N, steps, cfg_strength, ode_method="euler") -> float:
        evals = _ode_evals(steps, _ode_method_id(ode_method))
        return float(_lib.lib().f5_sample_flops(self.engine()["handle"], B, N, evals, float(cfg_strength)))

    # -- the reference's operator signature (dit.py:319-330 / unett.py:244-255) ----------------------------------
    @torch.no_grad()
    def forward(self, x, cond, text, time, mask=None, drop_audio_cond=False, drop_text=False, cfg_infer=False,
                cache=False):
        """Flow prediction: float[b | 2b, n, mel].  cfg_infer packs (cond, uncond) on the batch axis."""
        if drop_audio_cond != drop_text:
            raise NotImplementedError("only the joint (audio+text) drop used by CFG inference is built")
        B, N, mel = x.shape
        dev = x.device
        t0 = float(time.reshape(-1)[0]) if torch.is_tensor(time) else float(time)
        y = x.detach().float().contiguous().clone()
        sc = cond.detach().float().contiguous()
        duration = None if mask is None else mask.sum(dim=1).to(torch.int32).contiguous()
        packed = cfg_infer or drop_text
        v = torch.empty((2 * B if packed else B, N, mel), device=dev, dtype=torch.float32)
        self.run(y, sc, text.to(torch.int64).contiguous(), [t0, t0 + 1.0], duration, 1.0 if packed else 0.0, None, v,
                 use_graph=False)
        if cfg_infer:
            return v.to(x.dtype)
        return (v[B:] if drop_text else v).to(x.dtype)


class DiT(_Backbone):
    """backbones/dit.py:170-192 constructor arguments; conv_layers / text_dim as in configs/F5TTS_*Base.yaml"""

    KIND = "DiT"


class UNetT(_Backbone):
    """backbones/unett.py:108-128"""

    KIND = "UNetT"


# ----------------------------------------------------------------------------------------------------------------
# mel front-end
# ----------------------------------------------------------------------------------------------------------------
_fb_cache: dict = {}


def _mel_filterbank(n_freqs, n_mels, sample_rate, device):
    """HTK triangular filters, norm=None == torchaudio.functional.melscale_fbanks (model/modules.py:91-101)"""
    key = (n_freqs, n_mels, sample_rate, str(device))
    if key not in _fb_cache:
        all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
        m_max = 2595.0 * math.log10(1.0 + (sample_rate / 2) / 700.0)
        m_pts = torch.linspace(0.0, m_max, n_mels + 2)
        f_pts = 700.0 * (10.0 ** (m_pts / 2595.0) - 1.0)
        f_diff = f_pts[1:] - f_pts[:-1]
        slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
        fb = torch.clamp(torch.min(-slopes[:, :-2] / f_diff[:-1], slopes[:, 2:] / f_diff[1:]), min=0.0)
        _fb_cache[key] = fb.contiguous().to(device)
    return _fb_cache[key]


class MelSpec(nn.Module):
    """model/modules.py:112-151 — wav float[b, nw] -> log-mel float[b, n_mels, 1 + nw // hop]"""

    def __init__(self, n_fft=1024, hop_length=256, win_length=1024, n_mel_channels=100, target_sample_rate=24_000,
                 mel_spec_type="vocos"):
        super().__init__()
        if mel_spec_type != "vocos":
            raise NotImplementedError("only the vocos mel front-end is on the B200 path (bigvgan: out of scope)")
        if (n_fft, hop_length, win_length) != (1024, 256, 1024):
            raise NotImplementedError("the STFT kernel is built for n_fft=1024, hop=256, win=1024")
        self.n_fft, self.hop_length, self.win_length = n_fft, hop_length, win_length
        self.n_mel_channels, self.target_sample_rate = n_mel_channels, target_sample_rate
        self.register_buffer("dummy", torch.tensor(0), persistent=False)

    def forward(self, wav: torch.Tensor, frames_last: bool = True) -> torch.Tensor:
        if wav.ndim == 3:
            wav = wav.squeeze(1)
        assert wav.ndim == 2
        if not wav.is_cuda:
            raise _lib.F5LibraryError("MelSpec runs on the B200 only: move the waveform to a CUDA device")
        wav = wav.float().contiguous()
        B, nw = wav.shape
        T = 1 + nw // self.hop_length
        fb = _mel_filterbank(self.n_fft // 2 + 1, self.n_mel_channels, self.target_sample_rate, wav.device)
        shape = (B, self.n_mel_channels, T) if frames_last else (B, T, self.n_mel_channels)
        out = torch.empty(shape, device=wav.device, dtype=torch.float32)
        stream = torch.cuda.current_stream(wav.device).cuda_stream
        with torch.cuda.device(wav.device):
            _lib.check(_lib.lib().f5_mel_spectrogram(wav.data_ptr(), B, nw, fb.data_ptr(), self.n_mel_channels,
                                                     out.data_ptr(), 0 if frames_last else 1, stream),
                       "f5_mel_spectrogram")
        return out


# ----------------------------------------------------------------------------------------------------------------
# sampler
# ----------------------------------------------------------------------------------------------------------------
class CFM(nn.Module):
    """model/cfm.py:34-81 constructor; only `sample` (inference) is on this path — `forward` (training loss) is not."""

    def __init__(self, transformer: nn.Module, sigma=0.0, odeint_kwargs: dict = dict(method="euler"),
                 audio_drop_prob=0.3, cond_drop_prob=0.2, num_channels=None, mel_spec_module: nn.Module | None = None,
                 mel_spec_kwargs: dict = dict(), frac_lengths_mask=(0.7, 1.0), vocab_char_map: dict | None = None):
        super().__init__()
        self.frac_lengths_mask = frac_lengths_mask
        self.mel_spec = default(mel_spec_module, MelSpec(**mel_spec_kwargs))
        self.num_channels = default(num_channels, self.mel_spec.n_mel_channels)
        self.audio_drop_prob, self.cond_drop_prob = audio_drop_prob, cond_drop_prob
        self.transformer = transformer
        self.dim = transformer.dim
        self.sigma = sigma
        method = odeint_kwargs.get("method", "euler")
        if method not in ("euler", "midpoint"):
            raise NotImplementedError(f"the fused CFG + ODE update kernel implements method='euler' (the shipped default) "
                                      f"and 'midpoint', not {method!r}")
        self.odeint_kwargs = odeint_kwargs
        self.vocab_char_map = vocab_char_map
        self.use_cuda_graph = True

    @property
    def device(self):
        return next(self.parameters()).device

    def forward(self, *a, **k):
        raise NotImplementedError("training (CFM.forward, cfm.py:231-302) is outside the B200 inference path")

    @torch.no_grad()
    def sample(self, cond, text, duration, *, lens=None, steps=32, cfg_strength=1.0, sway_sampling_coef=None,
               seed: int | None = None, max_duration=65536, vocoder: Callable | None = None, use_epss=True,
               no_ref_audio=False, duplicate_test=False, t_inter=0.1, edit_mask=None, y0: torch.Tensor | None = None,
               exact_varlen: bool = False):
        """model/cfm.py:83-229.  Extra keywords: `y0` injects the initial noise (parity tests, SURVEY.md §8c);
        `exact_varlen=True` (batch > 1) computes every sample exactly as if it were alone in the batch with its own
        duration — the result of a loop of single-sample calls, in one batched call (f5_sample_args.exact_varlen)."""
        if self.training:  # (an unconditional eval() walks ~1800 sub-modules: 2 ms of host time per call)
            self.eval()
        if cond.ndim == 2:  # raw wave -> mel [b, n, d]
            cond = self.mel_spec(cond, frames_last=False)
            assert cond.shape[-1] == self.num_channels
        dtype = next(self.parameters()).dtype
        cond = cond.to(dtype)
        batch, cond_seq_len, device = *cond.shape[:2], cond.device
        if not exists(lens):
            lens = torch.full((batch,), cond_seq_len, device=device, dtype=torch.long)

        if isinstance(text, list):
            if exists(self.vocab_char_map):
                text = list_str_to_idx(text, self.vocab_char_map).to(device)
            else:
                text = list_str_to_tensor(text).to(device)
            assert text.shape[0] == batch

        cond_mask = lens_to_mask(lens)
        if edit_mask is not None:
            cond_mask = cond_mask & edit_mask
        if isinstance(duration, int):
            duration = torch.full((batch,), duration, device=device, dtype=torch.long)
        duration = torch.maximum(torch.maximum((text != -1).sum(dim=-1), lens) + 1, duration)
        duration = duration.clamp(max=max_duration)
        # the one host sync the reference also has (cfm.py:139); the largest token id rides along so that an id outside
        # the embedding table raises here, like the reference's nn.Embedding does (dit.py:103), instead of being read
        # out of bounds on the device
        n_frames, max_id = torch.stack([duration.amax(), text.amax().to(duration.dtype)]).tolist()
        if max_id >= self.transformer.text_num_embeds:
            raise IndexError(f"text token id {max_id} is outside the embedding table "
                             f"(text_num_embeds = {self.transformer.text_num_embeds})")

        if duplicate_test:
            test_cond = F.pad(cond, (0, 0, cond_seq_len, n_frames - 2 * cond_seq_len), value=0.0)
        cond = F.pad(cond, (0, 0, 0, n_frames - cond_seq_len), value=0.0)
        if no_ref_audio:
            cond = torch.zeros_like(cond)
        cond_mask = F.pad(cond_mask, (0, n_frames - cond_mask.shape[-1]), value=False).unsqueeze(-1)
        step_cond = torch.where(cond_mask, cond, torch.zeros_like(cond))
        dur32 = duration.to(torch.int32).contiguous() if batch > 1 else None  # `mask` of cfm.py:155-158

        if y0 is None:  # same RNG calls as cfm.py:196-201
            rows = []
            for dur in duration:
                if exists(seed):
                    torch.manual_seed(seed)
                rows.append(torch.randn(int(dur), self.num_channels, device=self.device, dtype=step_cond.dtype))
            y0 = pad_sequence(rows, padding_value=0, batch_first=True)
        t_start = 0
        if duplicate_test:
            t_start = t_inter
            y0 = (1 - t_start) * y0 + t_start * test_cond
            steps = int(steps * (1 - t_start))
        # time grid in fp32 (the reference builds it in the parameter dtype, i.e. fp16 on GPU: cfm.py:211-216)
        if t_start == 0 and use_epss:
            t = get_epss_timesteps(steps, device="cpu", dtype=torch.float32)
        else:
            t = torch.linspace(t_start, 1, steps + 1, dtype=torch.float32)
        if sway_sampling_coef is not None:
            t = t + sway_sampling_coef * (torch.cos(torch.pi / 2 * t) - 1 + t)

        y = y0.float().contiguous().clone()
        trajectory = torch.empty((steps + 1, batch, n_frames, self.num_channels), device=device, dtype=torch.float32)
        self.transformer.run(y, step_cond.float().contiguous(), text.to(torch.int64).contiguous(), t.tolist(), dur32,
                             cfg_strength, trajectory=trajectory, use_graph=self.use_cuda_graph,
                             exact_varlen=exact_varlen, ode_method=self.odeint_kwargs.get("method", "euler"))
        self.transformer.clear_cache()

        out = torch.where(cond_mask, cond, trajectory[-1].to(dtype))
        if exists(vocoder):
            out = vocoder(out.permute(0, 2, 1))
        return out, trajectory.to(dtype)
