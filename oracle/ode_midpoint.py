"""TEST INFRASTRUCTURE ONLY — torchdiffeq's fixed-grid midpoint solver for the CPU oracle and the reference.

The reference picks the ODE solver of ``CFM.sample`` through ``odeint_kwargs`` (cfm.py:39-42,218) and names
``"midpoint"`` as the alternative to Euler.  torchdiffeq is not installed here, so its fixed-grid midpoint method is
restated from the published algorithm (``Midpoint._step_func``: the increment of one step is
``dt * f(t0 + dt/2, y0 + f(t0, y0) * dt/2)``; only the caller's grid points are returned) and is **parity unpinned**
like the Euler restatement in ``oracle/ref_shims.py``.

* ``odeint`` — drop-in ``torchdiffeq.odeint`` for the reference: Euler is ``ref_shims._odeint`` unchanged.
* ``import_reference()`` — the unmodified reference imported with ``odeint`` registered as ``torchdiffeq.odeint``.
* ``sample(..., method=)`` — ``oracle.f5_oracle.sample`` (cfm.py:83-229) with the solver chosen; Euler is that function.

Used by ``oracle/make_golden_midpoint.py`` and the midpoint tests; the product package never imports it.
"""
from __future__ import annotations

import sys

import torch
import torch.nn.functional as F

from oracle import f5_oracle as O
from oracle import ref_shims

METHODS = ("euler", "midpoint")


def _check(method):
    if method not in METHODS:
        raise NotImplementedError(f"the oracle restates method='euler' and 'midpoint' only (got {method!r})")


def odeint(func, y0, t, *, method="euler", **kw):
    """torchdiffeq.odeint on the caller's grid t[0..S] with the fixed-grid "euler" or "midpoint" method."""
    _check(method)
    if method == "euler":
        return ref_shims._odeint(func, y0, t, method=method, **kw)
    ys = [y0]
    y = y0
    for k in range(t.shape[0] - 1):
        t0, t1 = t[k], t[k + 1]
        dt = t1 - t0
        half_dt = 0.5 * dt
        f0 = func(t0, y)
        y_mid = y + f0 * half_dt
        y = y + dt * func(t0 + half_dt, y_mid)
        ys.append(y)
    return torch.stack(ys, dim=0)


def import_reference():
    """ref_shims.import_reference() with this module's odeint as torchdiffeq.odeint (registered before the reference's
    cfm.py binds it with `from torchdiffeq import odeint`)."""
    td = sys.modules.get("torchdiffeq")
    if td is None:
        ref_shims._stub("torchdiffeq", odeint=odeint)
    elif td.odeint is not odeint:
        raise RuntimeError("torchdiffeq was registered before oracle.ode_midpoint: import the reference through "
                           "ode_midpoint.import_reference() in a fresh process")
    return ref_shims.import_reference()


@torch.no_grad()
def sample(sd, cfg: O.ArchConfig, cond, text, duration, *, lens=None, steps=32, cfg_strength=1.0,
           sway_sampling_coef=None, seed=None, max_duration=65536, use_epss=True, no_ref_audio=False,
           edit_mask=None, y0=None, method="midpoint") -> O.SampleResult:
    """oracle.f5_oracle.sample (model/cfm.py:83-229) with odeint_kwargs=dict(method=method)."""
    _check(method)
    kw = dict(lens=lens, steps=steps, cfg_strength=cfg_strength, sway_sampling_coef=sway_sampling_coef, seed=seed,
              max_duration=max_duration, use_epss=use_epss, no_ref_audio=no_ref_audio, edit_mask=edit_mask, y0=y0)
    if method == "euler":
        return O.sample(sd, cfg, cond, text, duration, **kw)
    # the prologue of f5_oracle.sample (cfm.py:103-216), then the solver
    if cond.ndim == 2:
        cond = O.mel_spectrogram(cond).permute(0, 2, 1)
    cond = cond.float()
    B, n_cond = cond.shape[:2]
    if lens is None:
        lens = torch.full((B,), n_cond, dtype=torch.long)
    cond_mask = O.lens_to_mask(lens)
    if edit_mask is not None:
        cond_mask = cond_mask & edit_mask
    if isinstance(duration, int):
        duration = torch.full((B,), duration, dtype=torch.long)
    duration = torch.maximum(torch.maximum((text != -1).sum(dim=-1), lens) + 1, duration).clamp(max=max_duration)
    N = int(duration.amax())
    cond = F.pad(cond, (0, 0, 0, N - n_cond), value=0.0)
    if no_ref_audio:
        cond = torch.zeros_like(cond)
    cond_mask = F.pad(cond_mask, (0, N - cond_mask.shape[-1]), value=False)[..., None]
    step_cond = torch.where(cond_mask, cond, torch.zeros_like(cond))
    mask = O.lens_to_mask(duration) if B > 1 else None
    if cfg.backbone == "DiT":
        seq_len = N if mask is None else mask.sum(dim=1)
        te = (O.text_embedding_dit(sd, cfg, text, seq_len, False), O.text_embedding_dit(sd, cfg, text, seq_len, True))
        fwd = O.dit_forward
    else:
        te = (O.text_embedding_unett(sd, cfg, text, N, False), O.text_embedding_unett(sd, cfg, text, N, True))
        fwd = O.unett_forward

    def fn(t, x):
        if cfg_strength < 1e-5:
            return fwd(sd, cfg, x, step_cond, te, t, mask, False)
        pred, null = fwd(sd, cfg, x, step_cond, te, t, mask, True).chunk(2, dim=0)
        return pred + (pred - null) * cfg_strength

    if y0 is None:
        rows = []
        for dur in duration.tolist():
            if seed is not None:
                torch.manual_seed(seed)
            rows.append(torch.randn(dur, cfg.mel_dim, dtype=torch.float32))
        y0 = torch.nn.utils.rnn.pad_sequence(rows, padding_value=0, batch_first=True)
    t = O.time_grid(steps, sway_sampling_coef, use_epss)
    traj = odeint(fn, y0, t, method=method)
    out = torch.where(cond_mask, cond, traj[-1])
    return O.SampleResult(out=out, trajectory=traj, y0=y0, t=t,
                          extras={"text_cond": te[0], "text_uncond": te[1], "mask": mask, "step_cond": step_cond})
