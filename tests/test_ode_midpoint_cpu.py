"""CPU: the midpoint ODE solver (odeint_kwargs=dict(method="midpoint"), cfm.py:39-42) on the host side.

  * the torchdiffeq restatement in oracle/ode_midpoint.py against the closed form of one step and its order of
    accuracy on an analytic linear ODE;
  * the oracle's midpoint sampler against vectors written by the UNMODIFIED reference through that restatement
    (tests/golden/*_midpoint.npz, oracle/make_golden_midpoint.py), bit for bit like test_oracle_vs_golden.py;
  * CFM / load_model accept and carry the method; every other method still raises.
"""
import ast
import math
import os

import numpy as np
import pytest
import torch

import f5_tts_b200 as F5
from f5_tts_b200 import infer
from oracle import f5_oracle as O
from oracle import ode_midpoint as M


def _lam(t):
    return torch.exp(-t) if torch.is_tensor(t) else math.exp(-t)


def _exact(y0, t):
    """y' = exp(-t) y  ->  y(t) = y0 exp(1 - exp(-t))  (the local error keeps one sign, so the order shows cleanly)"""
    return y0 * torch.exp(1.0 - torch.exp(-t))


def _solve(method, steps, y0):
    t = torch.linspace(0.0, 1.0, steps + 1, dtype=torch.float64)
    return M.odeint(lambda tt, y: _lam(tt) * y, y0, t, method=method)


def test_shim_euler_is_the_existing_restatement():
    from oracle import ref_shims

    y0 = torch.tensor([1.0, 0.3], dtype=torch.float64)
    t = torch.linspace(0.0, 1.0, 9, dtype=torch.float64)
    f = lambda tt, y: _lam(tt) * y  # noqa: E731
    assert torch.equal(M.odeint(f, y0, t, method="euler"), ref_shims._odeint(f, y0, t))


def test_shim_midpoint_one_step_closed_form():
    y0 = torch.tensor([1.0, -0.5, 2.0], dtype=torch.float64)
    t0, t1 = 0.2, 0.45
    t = torch.tensor([t0, t1], dtype=torch.float64)
    traj = M.odeint(lambda tt, y: _lam(tt) * y, y0, t, method="midpoint")
    dt = t1 - t0
    lam0, lamh = _lam(t0), _lam(t0 + dt / 2)
    want = y0 + dt * lamh * (y0 + dt / 2 * lam0 * y0)
    assert traj.shape == (2, 3)
    assert torch.equal(traj[0], y0)
    assert torch.allclose(traj[1], want, rtol=1e-14, atol=0)


def test_shim_midpoint_is_second_order_euler_first():
    y0 = torch.tensor([1.0, 0.3], dtype=torch.float64)
    exact = _exact(y0, torch.tensor(1.0, dtype=torch.float64))
    err = {m: [float((_solve(m, n, y0)[-1] - exact).abs().max()) for n in (8, 16, 32, 64)] for m in ("euler", "midpoint")}
    ratios = {m: [a / b for a, b in zip(e, e[1:])] for m, e in err.items()}
    print("error ratios per doubling of steps:", ratios)
    assert all(r >= 3.5 for r in ratios["midpoint"])
    assert all(1.7 <= r <= 2.3 for r in ratios["euler"])
    assert err["midpoint"][-1] < err["euler"][-1] / 100


def test_shim_keeps_only_grid_points():
    y0 = torch.ones(2, 4, dtype=torch.float64)
    calls = []

    def f(t, y):
        calls.append(float(t))
        return -y

    t = torch.tensor([0.0, 0.25, 1.0], dtype=torch.float64)
    traj = M.odeint(f, y0, t, method="midpoint")
    assert traj.shape == (3, 2, 4)
    assert calls == [0.0, 0.125, 0.25, 0.625]


@pytest.mark.parametrize("name", ["dit_tiny_b1_midpoint", "dit_tiny_b3_midpoint"])
def test_oracle_midpoint_vs_reference(golden_dir, name):
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    assert str(z["method"]) == "midpoint"
    body = str(z["cfg"])
    body = body[body.index("(") + 1: body.rindex(")")]
    cfg = O.ArchConfig(**{k: ast.literal_eval(v) for k, v in (p.split("=") for p in body.split(", "))})
    sd = O.synthetic_state_dict(cfg, seed=int(z["wseed"]))
    dur = z["duration"]
    duration = int(dur) if dur.ndim == 0 else torch.from_numpy(dur).long()
    lens = torch.from_numpy(z["lens"]).long() if z["lens"].size else None
    sway = None if np.isnan(z["sway"]) else float(z["sway"])
    res = M.sample(sd, cfg, torch.from_numpy(z["cond"]), torch.from_numpy(z["text"]), duration, lens=lens,
                   steps=int(z["steps"]), cfg_strength=float(z["cfg_strength"]), sway_sampling_coef=sway,
                   seed=int(z["seed"]), method="midpoint")
    assert res.trajectory.shape[0] == int(z["steps"]) + 1
    assert torch.equal(res.y0, torch.from_numpy(z["y0"]))
    for got, key in ((res.trajectory[1], "traj_1"), (res.trajectory[-1], "traj_last"), (res.out, "out")):
        want = torch.from_numpy(z[key])
        assert float((got - want).norm() / want.norm()) == 0.0, key
    # the solver matters at these step counts: Euler on the same grid lands elsewhere
    eul = M.sample(sd, cfg, torch.from_numpy(z["cond"]), torch.from_numpy(z["text"]), duration, lens=lens,
                   steps=int(z["steps"]), cfg_strength=float(z["cfg_strength"]), sway_sampling_coef=sway,
                   seed=int(z["seed"]), method="euler")
    assert float((eul.out - res.out).norm() / res.out.norm()) > 1e-3


def _tiny_dit():
    return F5.DiT(dim=128, depth=1, heads=2, ff_mult=2, text_dim=64, conv_layers=1, text_num_embeds=10)


def test_cfm_accepts_midpoint():
    m = F5.CFM(transformer=_tiny_dit(), odeint_kwargs=dict(method="midpoint"))
    assert m.odeint_kwargs["method"] == "midpoint"
    assert F5.CFM(transformer=_tiny_dit()).odeint_kwargs["method"] == "euler"


@pytest.mark.parametrize("method", ["rk4", "dopri5", "heun3"])
def test_other_methods_still_raise(method):
    with pytest.raises(NotImplementedError, match=method):
        F5.CFM(transformer=_tiny_dit(), odeint_kwargs=dict(method=method))
    with pytest.raises(NotImplementedError):
        M.sample(None, None, None, None, None, method=method)
    with pytest.raises(NotImplementedError):
        M.odeint(None, None, None, method=method)


def test_load_model_forwards_ode_method(golden_dir):
    arch = dict(dim=128, depth=1, heads=2, ff_mult=2, text_dim=64, conv_layers=1, text_mask_padding=False,
                pe_attn_head=1)
    m = infer.load_model(F5.DiT, arch, "", vocab_file=os.path.join(golden_dir, "vocab.txt"), ode_method="midpoint",
                         device="cpu")
    assert isinstance(m, F5.CFM) and m.odeint_kwargs == dict(method="midpoint")
    with pytest.raises(NotImplementedError):
        infer.load_model(F5.DiT, arch, "", vocab_file=os.path.join(golden_dir, "vocab.txt"), ode_method="rk4",
                         device="cpu")
