"""The optimisers of `--optimiser` besides Adam (pixray.py:536-553): the CPU restatements in tests/optim_ref.py against
torch.optim, DiffGrad against its update rule worked by hand, and the api's choice of optimiser per drawer and per
rebuild against a recording engine."""
import json
import math
import os

import numpy as np
import pytest
import torch

from fake_engine import FakeEngine
from optim_ref import STATES
from pixray_b200 import api
from pixray_b200 import engine as E

TORCH_OPTIM = {"Adam": torch.optim.Adam, "AdamW": torch.optim.AdamW, "Adagrad": torch.optim.Adagrad,
               "Adamax": torch.optim.Adamax}


def _grads(n, shape, seed):
    """Seeded gradients with exact zeros and entries that flip sign every step."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for k in range(n):
        x = torch.randn(shape, generator=g) * (0.1 + k % 3)
        x[..., 0, :] = 0.0
        x[..., 1, :] = (-1.0) ** k * 0.5
        x[..., 2, :3] = (-1.0) ** (k // 2) * 1e-6
        out.append(x)
    return out


@pytest.mark.parametrize("name", sorted(TORCH_OPTIM))
def test_oracle_matches_torch_optim(name):
    shape, lr = (1, 256, 16, 16), 0.2
    z0 = torch.randn(shape, generator=torch.Generator().manual_seed(1))
    grads = _grads(10, shape, 2)
    p = torch.nn.Parameter(z0.clone())
    opt = TORCH_OPTIM[name]([p], lr=lr)
    z, st = z0.clone(), STATES[name](z0)
    cur_lr, worst = lr, 0.0
    for k, g in enumerate(grads):
        if k == 5:  # a rebuild at lr / 10 (rebuild_optimisers after a drop): fresh state on both sides
            cur_lr = lr / 10
            opt = TORCH_OPTIM[name]([p], lr=cur_lr)
            st = STATES[name](z)
        p.grad = g.clone()
        opt.step()
        z = st.step(z, g, cur_lr)
        worst = max(worst, (z - p.detach()).abs().max().item())
    print(f"[optim] {name} oracle vs torch.optim: max_abs_err {worst:.3e}")
    assert worst <= 1e-6


def _diffgrad_by_hand(z, grads, lr, b1=0.9, b2=0.999, eps=1e-8):
    m = v = p = 0.0
    for t, g in enumerate(grads, start=1):
        m = b1 * m + (1 - b1) * g
        v = b2 * v + (1 - b2) * g * g
        denom = math.sqrt(v) + eps
        dfc = 1.0 / (1.0 + math.exp(-abs(p - g)))
        p = g
        z = z - lr * math.sqrt(1 - b2 ** t) / (1 - b1 ** t) * (m * dfc) / denom
    return z


def test_diffgrad_oracle_follows_the_rule_by_hand():
    z0 = torch.tensor([0.5, -1.25, 2.0, 0.0, 0.3], dtype=torch.float32)
    steps = [torch.tensor(r, dtype=torch.float32) for r in ([0.3, -2.0, 0.0, 1e-3, 5.0],
                                                             [-0.4, -2.0, 0.7, 1e-3, -5.0],
                                                             [0.1, 3.0, 0.0, -2e-3, 5.0])]
    st = STATES["DiffGrad"](z0)
    z = z0.clone()
    for g in steps:
        z = st.step(z, g, 0.2)
    for i in range(z0.numel()):
        want = _diffgrad_by_hand(float(z0[i]), [float(g[i]) for g in steps], 0.2)
        assert abs(float(z[i]) - want) <= 1e-6 * max(1.0, abs(want)), (i, float(z[i]), want)


def test_diffgrad_friction_is_one_half_when_the_gradient_repeats():
    z = torch.randn(64, generator=torch.Generator().manual_seed(3))
    g = torch.randn(64, generator=torch.Generator().manual_seed(4))
    st = STATES["DiffGrad"](z)
    z = st.step(z, g, 0.1)
    assert not torch.all(st.dfc == 0.5)  # the first step compares with a zero previous gradient
    st.step(z, g.clone(), 0.1)
    assert torch.all(st.dfc == 0.5)


# ------------------------------------------------------------------ api: which optimiser is built when
def test_apply_settings_accepts_the_new_optimisers():
    for name in ("AdamW", "Adagrad", "Adamax", "DiffGrad"):
        api.reset_settings()
        api.add_settings(prompts="x", optimiser=name)
        assert api.apply_settings().optimiser == name
    api.reset_settings()


@pytest.mark.parametrize("name", ["AdamP", "RAdam", "adam"])
def test_adamp_and_unknown_optimisers_are_still_refused(name):
    api.reset_settings()
    api.add_settings(prompts="x", optimiser=name)
    with pytest.raises(NotImplementedError):
        api.apply_settings()
    api.reset_settings()


class OptimiserRecordingEngine(FakeEngine):
    """FakeEngine plus the optimiser switch of B200Engine."""

    def __init__(self, **kw):
        super().__init__(**kw)
        self.optimizer = "Adam"

    def set_optimizer(self, name):
        assert name in E.OPTIMISERS
        self.optimizer = name
        self._log("set_optimizer", kind=name)


@pytest.fixture
def rec(monkeypatch):
    monkeypatch.setattr(api, "_engine_factory", OptimiserRecordingEngine)
    FakeEngine.loss_script = staticmethod(lambda it, n: np.full(n, 1.0 / (1 + it), dtype=np.float32))
    api.reset_settings()
    yield
    api.reset_settings()


def _run(tmp_path, **kw):
    (tmp_path / "vectors").mkdir(exist_ok=True)
    (tmp_path / "vectors" / "textoff.json").write_text(json.dumps({"ViT-B/16": [[0.1] * 512]}))
    os.environ["PIXRAY_ROOT"] = str(tmp_path)
    base = dict(prompts="x", size=[64, 64], num_cuts=8, outdir="", seed="7", clip_models="ViT-B/16",
                b200_allow_synthetic=True)
    base.update(kw)
    api.add_settings(**base)
    args = api.apply_settings()
    api.do_init(args)
    assert api.do_run(args) is True
    return api._state.engine


def _opt_calls(eng):
    """The optimiser calls in order, each tagged with the number of iterations issued before it."""
    out, its = [], 0
    for name, kw in eng.calls:
        if name == "iterate":
            its += 1
        elif name == "set_optimizer":
            out.append((its, kw["kind"]))
        elif name == "reset_optimizer":
            out.append((its, "reset"))
    return out


def test_vqgan_adamw_host_mode_with_a_scheduled_drop(rec, tmp_path):
    eng = _run(tmp_path, optimiser="AdamW", iterations=20, learning_rate_drops=[50], b200_device_checkdrop=False)
    assert not api._state.managed
    # AdamW at init; the drop after iteration 9 rebuilds the same kind, which is a reset
    assert _opt_calls(eng) == [(0, "AdamW"), (10, "reset")]
    lrs = [round(c[1]["lr"], 6) for c in eng.calls if c[0] == "iterate"]
    assert lrs == [0.2] * 10 + [0.02] * 10


def test_fft_ignores_the_optimiser_setting(rec, tmp_path):
    eng = _run(tmp_path, drawer="fft", optimiser="DiffGrad", iterations=4, learning_rate_drops=None)
    assert "set_optimizer" not in eng.names()  # FftDrawer.get_opts builds its own Adam (fftdrawer.py:63-67)
    assert _opt_calls(eng) == [(0, "reset")]


def test_vdiff_switches_to_adam_from_the_second_step_on(rec, tmp_path):
    sd = {"dummy": torch.zeros(1)}
    eng = _run(tmp_path, drawer="vdiff", optimiser="Adagrad", iterations=5, learning_rate_drops=None,
               b200_weights={"vdiff": sd})
    # iteration 0 steps Adagrad; from iteration 1 on the loop installs a fresh Adam after every step, and once more in
    # the final call that only checks in (pixray.py:1489-1495)
    assert _opt_calls(eng) == [(0, "Adagrad"), (2, "Adam"), (3, "reset"), (4, "reset"), (5, "reset"), (5, "reset")]


def test_vdiff_drop_rebuild_installs_the_chosen_optimiser_again(rec, tmp_path):
    sd = {"dummy": torch.zeros(1)}
    eng = _run(tmp_path, drawer="vdiff", optimiser="Adagrad", iterations=6, learning_rate_drops=[50],
               b200_weights={"vdiff": sd})
    # drop at iteration 2: the vdiff branch's fresh Adam, then rebuild_optimisers' Adagrad for iteration 3, which the
    # vdiff branch replaces with Adam again after it
    assert _opt_calls(eng) == [(0, "Adagrad"), (2, "Adam"), (3, "reset"), (3, "Adagrad"), (4, "Adam"), (5, "reset"),
                               (6, "reset"), (6, "reset")]


def test_default_adam_run_never_switches(rec, tmp_path):
    eng = _run(tmp_path, iterations=20, learning_rate_drops=[50, 25])
    assert "set_optimizer" not in eng.names()
    assert eng.names().count("reset_optimizer") == 3
