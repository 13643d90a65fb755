"""GPU checks of the optimiser kinds (pxr_set_optimizer): the plain and the device-managed step against the CPU
restatements (oracle/ref_path.py's AdamState, tests/optim_ref.py) followed by clip_z, checkpoints that carry DiffGrad's
extra state, and pixray.run() end to end with each new optimiser.

Bound for every update: max |z_engine - z_oracle| <= 2e-6 * max(1, max |z|) -- fp32 on both sides, the engine with
different but exactly rounded groupings (sqrt(v) * (1 / sqrt(bc2)) instead of sqrt(v) / sqrt(bc2)), so the difference is a
few ulp of z."""
import numpy as np
import pytest
import torch

from oracle import ref_path as R
from optim_ref import STATES
from pixray_b200 import engine as E
from test_pipeline_gpu import SMALL_CLIP, build

pytestmark = pytest.mark.gpu

KINDS = list(E.OPTIMISERS)
STATE_HEADER_BYTES = 64  # pxr_save_state's header: magic, version, z_numel, 4 int32 counters, DropState


def _bound(z):
    return 2e-6 * max(1.0, z.abs().max().item())


def _pixel_engine(seed=0, grid=(8, 8)):
    clip = R.init_clip_weights(R.ClipVisual(224, SMALL_CLIP["patch"], SMALL_CLIP["width"], SMALL_CLIP["layers"],
                                            SMALL_CLIP["heads"], SMALL_CLIP["out_dim"]), seed + 1)
    eng = E.B200Engine(drawer=E.DRAWER_PIXEL, image_hw=(32, 32), grid=grid, cutn=8, clip=[SMALL_CLIP], noise_fac=0.1,
                       seed=seed)
    eng.load_module(E.MOD_CLIP0, clip.state_dict())
    eng.finalize()
    g = torch.Generator().manual_seed(seed + 2)
    z = (torch.rand(1, 3, *grid, generator=g) * 1.4 - 0.2).contiguous()  # some colours outside [0, 1]
    return eng, z, lambda x: x.clamp(0, 1)  # FastPixelDrawer.clip_z (fast_pixeldrawer.py:98-100)


def _vqgan_engine(seed):
    vq, _, eng, _, z = build(cutn=8, seed=seed)
    zmin, zmax = R.vqgan_z_bounds(vq)
    return eng, z, lambda x: torch.maximum(torch.minimum(x, zmax), zmin)  # VqganDrawer.clip_z (vqgan.py:202-204)


def _grad(shape, k, scale, seed):
    g = torch.randn(shape, generator=torch.Generator().manual_seed(seed + k)) * scale
    g[..., 0, :] = 0.0                             # exact zeros
    g[..., 1, :] = (-1.0) ** k * 0.5 * scale       # sign flips every step
    return g.contiguous()


@pytest.mark.parametrize("drawer", ["vqgan", "pixel"])
@pytest.mark.parametrize("kind", KINDS)
def test_plain_step_matches_the_oracle(kind, drawer):
    """pxr_step with set_z_grad: steps 0-3 at lr, a reset at lr / 10 for steps 4-5 (fresh state of the same kind), then a
    switch to the next kind for steps 6-7 (fresh state of that kind)."""
    eng, z, clip_z = _vqgan_engine(31) if drawer == "vqgan" else _pixel_engine(3)
    scale = 1e-2 if drawer == "vqgan" else 1e-3
    eng.synth(z.cuda())  # loads z into the engine
    eng.set_optimizer(kind)
    cur, lr = kind, 0.2
    st = STATES[cur](z)
    z_ref, worst = z.clone(), 0.0
    out = torch.empty(z.shape, device="cuda")
    for k in range(8):
        if k == 4:
            lr /= 10
            eng.reset_optimizer()
            st = STATES[cur](z_ref)
        if k == 6:
            cur = KINDS[(KINDS.index(kind) + 1) % len(KINDS)]
            eng.set_optimizer(cur)
            st = STATES[cur](z_ref)
        g = _grad(z.shape, k, scale, 100)
        eng.set_z_grad(g.cuda())
        eng.step(out, lr, k)
        z_ref = clip_z(st.step(z_ref, g, lr))
        err = (out.cpu() - z_ref).abs().max().item()
        worst = max(worst, err)
        assert err <= _bound(z_ref), (k, cur, err)
    moved = (z_ref - clip_z(z)).abs().max().item()
    print(f"[optim] plain step {kind}->{cur} on {drawer}: max |dz| {worst:.3e} (bound {_bound(z_ref):.1e}, moved {moved:.2e})")
    assert moved > 10 * _bound(z_ref)


@pytest.mark.parametrize("kind", KINDS)
def test_managed_step_matches_the_oracle(kind):
    """The device-managed step (checkdrop, scheduled drop at iteration 3) applies the chosen optimiser, and the drop leaves a
    fresh instance of the same kind at lr / 10 behind."""
    vq, _, eng, _, z = build(cutn=8, seed=17)
    zmin, zmax = R.vqgan_z_bounds(vq)
    eng.set_optimizer(kind)
    eng.set_schedule(0.05, iter_drop_delay=12, max_loss_drops=1, auto_stop=False, drops=[3])
    st, lr = STATES[kind](z), 0.05
    za = z.clone().cuda()
    worst, rebuilt = 0.0, []
    for it in range(6):
        z0 = za.cpu()
        eng.iterate(za, 0.0, it)
        eng.sync()
        g = eng.debug_read("z_grad", z.shape).cpu()
        rec = eng.poll_status()
        assert rec is not None and rec["iter"] == it and not rec["stopped"]
        want = torch.maximum(torch.minimum(st.step(z0, g, lr), zmax), zmin)
        err = (za.cpu() - want).abs().max().item()
        worst = max(worst, err)
        assert err <= _bound(want), (it, err)
        if rec["rebuilt"]:
            rebuilt.append(it)
            st = STATES[kind](z)
        lr = rec["lr"]
    assert rebuilt == [3] and abs(lr - 0.005) < 1e-9
    print(f"[optim] managed step {kind}: max |dz| {worst:.3e}")


def test_checkpoint_carries_the_diffgrad_state():
    """A DiffGrad session saved at iteration 3, restored into a fresh engine and continued, follows the uninterrupted one
    (same bulk criterion as the Adam checkpoint test: the last bits of the gradients differ run to run)."""
    _, _, eng_a, _, z = build(cutn=8, seed=23)
    _, _, eng_b, _, _ = build(cutn=8, seed=23)
    n = z.numel()
    assert len(eng_a.save_state()) == STATE_HEADER_BYTES + 3 * n * 4  # Adam: the format blobs always had
    for e in (eng_a, eng_b):
        e.set_optimizer("DiffGrad")
        e.set_schedule(0.05, iter_drop_delay=12, max_loss_drops=2, auto_stop=False, drops=[1])
    za = z.clone().cuda()
    for it in range(3):
        eng_a.iterate(za, 0.0, it)
    eng_a.sync()
    blob = eng_a.save_state()
    assert len(blob) == STATE_HEADER_BYTES + 4 * n * 4  # + the previous gradient
    for it in range(3, 7):
        eng_a.iterate(za, 0.0, it)
    eng_a.sync()
    eng_b.load_state(blob)
    zb = eng_b.read_z()
    for it in range(3, 7):
        eng_b.iterate(zb, 0.0, it)
    eng_b.sync()
    ra, rb = eng_a.poll_status(), eng_b.poll_status()
    assert ra["num_loss_drop"] == rb["num_loss_drop"] == 1 and abs(ra["lr"] - rb["lr"]) < 1e-9
    moved = (za - z.cuda()).abs().max().item()
    diff = (za - zb).abs()
    print(f"[optim] DiffGrad resume: moved {moved:.3e}, median diff {diff.median().item():.3e}")
    assert moved > 0.02 and diff.median().item() < 1e-3 * moved and (diff > 0.1 * moved).float().mean().item() < 0.02
    # without the previous gradient the continuation would differ: a DiffGrad blob does not load into an Adam engine
    _, _, eng_c, _, _ = build(cutn=8, seed=23)
    with pytest.raises(E.EngineError, match="DiffGrad.*Adam"):
        eng_c.load_state(blob)


def _api_run(drawer, optimiser, **kw):
    from pixray_b200 import api
    api.reset_settings()
    api.add_settings(prompts="a cat", drawer=drawer, optimiser=optimiser, clip_models="ViT-B/16", outdir="",
                     vector_prompts="none", b200_allow_synthetic=True, seed="3", **kw)
    args = api.apply_settings()
    api.do_init(args)
    z0 = api._state.drawer.get_z_copy().float().cpu()
    api.do_run(args)
    img = api.get_image()
    z1 = api._state.drawer.get_z().detach().float().cpu()
    assert img is not None and torch.isfinite(img).all()
    assert np.isfinite(api._state.losses).all() and torch.isfinite(z1).all()
    moved = (z1 - z0).abs().max().item()
    print(f"[optim] api.run {drawer} {optimiser} {kw}: z moved {moved:.3e}, losses {api._state.losses}")
    assert moved > 0
    api.reset_settings()


@pytest.mark.parametrize("checkdrop", [True, False])
@pytest.mark.parametrize("optimiser", ["AdamW", "Adagrad", "Adamax", "DiffGrad"])
def test_api_run_vqgan(optimiser, checkdrop):
    _api_run("vqgan", optimiser, size=[128, 128], num_cuts=8, iterations=20, learning_rate_drops=[50],
             b200_device_checkdrop=checkdrop)


def test_api_run_pixel_and_vdiff():
    _api_run("pixel", "Adamax", size=[64, 64], num_cuts=8, iterations=10)
    _api_run("vdiff", "DiffGrad", size=[64, 64], num_cuts=8, iterations=4, learning_rate_drops=None)
