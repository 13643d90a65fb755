"""The module-level entry points (pixray_b200/api.py = pixray.py:2005-2124) on the CPU: the settings pipeline against what
the real reference resolves (tests/golden/api_settings.json, oracle/make_golden_api.py), and the do_init / do_run control flow
(prompt order, learning-rate drops, auto-stop, vdiff re-noising) against a recording stand-in for the engine."""
import json
import os

import numpy as np
import pytest
import torch

from fake_engine import FakeEngine
from pixray_b200 import api
from pixray_b200 import engine as E
from pixray_b200 import plugins as P

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "api_settings.json")))


@pytest.fixture
def fake(monkeypatch):
    monkeypatch.setattr(api, "_engine_factory", FakeEngine)
    FakeEngine.loss_script = staticmethod(lambda it, n: np.full(n, 1.0 / (1 + it), dtype=np.float32))
    api.reset_settings()
    yield
    api.reset_settings()


@pytest.mark.parametrize("name", sorted(GOLD))
def test_settings_resolve_like_the_reference(name):
    case = GOLD[name]
    api.reset_settings()
    api.add_settings(outdir="", **case["settings"])
    a = api.apply_settings()
    for k, want in case["want"].items():
        assert getattr(a, k) == want, (name, k, getattr(a, k), want)
    assert api.get_settings()["outdir"] == ""


def test_unknown_setting_and_unknown_plugins_raise():
    api.reset_settings()
    api.add_settings(prompts="x", bogus=1)
    with pytest.raises(ValueError, match="Requested setting not found, aborting: bogus=1"):   # pixray.py:2093
        api.apply_settings()
    api.reset_settings()
    api.add_settings(prompts="x", drawer="clipdraw")
    with pytest.raises(ValueError):
        api.apply_settings()
    api.reset_settings()
    api.add_settings(prompts="x", custom_loss="style")
    with pytest.raises(ValueError, match="Requested loss not found"):
        api.apply_settings()
    api.reset_settings()


@pytest.mark.parametrize("kw", [dict(target_images="t.png"), dict(optimiser="AdamP"),
                                dict(perceptors="slip"), dict(make_video=True),
                                dict(animation_dir="anim"), dict(transparent=True)])
def test_options_off_the_hot_path_are_refused_not_ignored(kw):
    api.reset_settings()
    api.add_settings(prompts="x", **kw)
    with pytest.raises(NotImplementedError):
        api.apply_settings()
    api.reset_settings()


def test_drawer_and_loss_options_are_contributed_by_the_plugins():
    api.reset_settings()
    api.add_settings(prompts="x", drawer="fft", fft_decay=2.0, custom_loss="smoothness:0.5", smoothness_type="log")
    a = api.apply_settings()
    assert a.fft_decay == 2.0 and a.fft_lrate == 0.3 and a.smoothness_type == "log"
    api.reset_settings()
    api.add_settings(prompts="x", fft_decay=2.0)          # not a vqgan option
    with pytest.raises(ValueError):
        api.apply_settings()
    api.reset_settings()


def _init(tmp_path, **kw):
    (tmp_path / "vectors").mkdir(exist_ok=True)
    (tmp_path / "vectors" / "textoff.json").write_text(json.dumps({"ViT-B/16": [[0.1] * 512], "ViT-B/32": [[0.2] * 512]}))
    os.environ["PIXRAY_ROOT"] = str(tmp_path)
    base = dict(size=[64, 64], num_cuts=8, outdir="", seed="7", b200_allow_synthetic=True)
    base.update(kw)
    api.add_settings(**base)
    args = api.apply_settings()
    return api.do_init(args)


def test_do_init_builds_the_session_in_the_reference_order(fake, tmp_path):
    args = _init(tmp_path, prompts="a cat:2|a dog:-0.5:0.3", clip_models="ViT-B/32,ViT-B/16", iterations=20,
                 noise_prompt_seeds=[3], noise_prompt_weights=[0.25])
    eng = api._state.engine
    assert eng.kw["image_hw"] == (64, 64) and eng.kw["cutn"] == 8 and len(eng.kw["clip"]) == 2
    assert eng.names()[:4] == ["load_module", "load_module", "load_module", "finalize"]
    # per perceptor: text prompts, then the vector prompt at 10 % weight; the noise prompt lands on the loop's last perceptor
    for i, name in enumerate(args.clip_models):
        emb, w, stops = eng.prompts[i]
        want_w = [2.0, -0.5, 0.1] + ([0.25] if i == 1 else [])
        assert w == pytest.approx(want_w)
        assert stops[1] == pytest.approx(0.3) and stops[0] == float("-inf")
        assert np.allclose(emb[2], 0.2 if name == "ViT-B/32" else 0.1)
    assert isinstance(api._state.drawer, P.VqganDrawer) and tuple(api._state.drawer.get_z().shape) == (1, 256, 4, 4)
    assert api._state.lr == pytest.approx(0.2) and eng.names().count("reset_optimizer") == 1
    # same seed string -> same starting latent (sha512 seed, pixray.py:595-606)
    z0 = api._state.drawer.get_z_copy()
    api.reset_settings()
    _init(tmp_path, prompts="a cat:2|a dog:-0.5:0.3", clip_models="ViT-B/32,ViT-B/16", iterations=20)
    assert torch.equal(z0, api._state.drawer.get_z())


def test_text_prompts_need_a_text_tower(fake, tmp_path):
    with pytest.raises(ValueError, match="text tower"):
        _init(tmp_path, prompts="a cat", clip_models="ViT-B/16", b200_allow_synthetic=False)
    api.reset_settings()
    seen = []

    def enc(model, txt):
        seen.append((model, txt))
        return torch.ones(1, 512)
    _init(tmp_path, prompts="a cat|a dog", clip_models="ViT-B/16", b200_allow_synthetic=False, b200_text_encoder=enc)
    assert seen == [("ViT-B/16", "a cat"), ("ViT-B/16", "a dog")]


def test_unbuilt_configurations_fail_loudly(fake, tmp_path):
    for kw in (dict(clip_models="RN50"),):
        api.reset_settings()
        with pytest.raises(NotImplementedError):
            _init(tmp_path, prompts="x", **kw)


def test_default_widescreen_aspect_reaches_the_engine(fake, tmp_path):
    """The reference's DEFAULT canvas is widescreen (aspect='widescreen', quality 'normal': 384 x 216, pixray.py:1753,
    1864-1878): global_aspect_width = 384 / 216 from the requested size, the VQGAN canvas rounds to 384 x 208."""
    args = _init(tmp_path, prompts="x", clip_models="ViT-B/16", size=None)
    assert args.size == [384, 216]
    eng = api._state.engine
    assert eng.kw["image_hw"] == (208, 384) and abs(eng.kw["cut_aspect"] - 384 / 216) < 1e-12
    assert abs(api._state.make_cutouts.aspect - 384 / 216) < 1e-12
    api.reset_settings()
    _init(tmp_path, prompts="x", clip_models="ViT-B/16", aspect="square", size=None)
    assert "cut_aspect" not in api._state.engine.kw and api._state.engine.kw["image_hw"] == (288, 288)


def test_batches_preset_reaches_the_engine(fake, tmp_path):
    """quality='best' means batches = 2 (pixray.py:1864-1878): two ascend_txt + backward passes per optimiser step."""
    args = _init(tmp_path, prompts="x", quality="best", clip_models="ViT-B/16", size=[128, 128])
    assert args.batches == 2
    assert ("set_batches", {"batches": 2}) in api._state.engine.calls


def test_do_run_scheduled_learning_rate_drops(fake, tmp_path):
    args = _init(tmp_path, prompts="x", clip_models="ViT-B/16", iterations=20, learning_rate_drops=[50, 25])
    assert args.learning_rate_drops == [9, 4]                      # percent of iterations - 1 (pixray.py:1999-2003)
    assert api.do_run(args) is True
    eng = api._state.engine
    its = [(c[1]["it"], round(c[1]["lr"], 6)) for c in eng.calls if c[0] == "iterate"]
    assert [i for i, _ in its] == list(range(20))                  # iterations 0..19, the 20th call only checks in
    # a drop takes effect AFTER the iteration that triggers it (rebuild_opts_when_done), each one divides by 10
    assert [lr for _, lr in its] == [0.2] * 5 + [0.02] * 5 + [0.002] * 10
    assert eng.names().count("reset_optimizer") == 3               # fresh Adam at init and at every drop
    assert api._state.cur_iteration == 20 and api.get_image() is not None
    assert eng.names()[-1] == "synth"                              # final checkin renders the image


def test_do_run_auto_stop_on_plateau(fake, tmp_path):
    # the loss stops improving at iteration 3: 12 iterations later (iter_drop_delay) checkdrop fires, auto_stop turns that
    # into a drop, and with one scheduled drop the second plateau ends the run (num_loss_drop > max_loss_drops)
    FakeEngine.loss_script = staticmethod(lambda it, n: np.full(n, max(1.0 - 0.1 * it, 0.7), dtype=np.float32))
    args = _init(tmp_path, prompts="x", clip_models="ViT-B/16", iterations=200, learning_rate_drops=[99], auto_stop=True)
    assert api.do_run(args) is True
    its = [(c[1]["it"], round(c[1]["lr"], 6)) for c in api._state.engine.calls if c[0] == "iterate"]
    # best at 3 -> drop after 15 (best_loss reset, pixray.py:1509-1510) -> new best at 16 -> second plateau ends the run at 28
    assert its[-1][0] == 28 and len(its) == 29
    assert [lr for _, lr in its] == [0.2] * 16 + [0.02] * 13


def test_return_display_hands_control_back(fake, tmp_path):
    args = _init(tmp_path, prompts="x", clip_models="ViT-B/16", iterations=50, display_every=20)
    assert api.do_run(args, return_display=True) is False and api._state.cur_iteration == 20
    assert api.do_run(args, return_display=True) is False and api._state.cur_iteration == 40
    assert api.do_run(args, return_display=True) is True and api._state.cur_iteration == 50


def test_runtime_errors_get_the_hint_and_propagate(fake, tmp_path, capsys):
    args = _init(tmp_path, prompts="x", clip_models="ViT-B/16", iterations=5)

    def boom(*a, **k):
        raise RuntimeError("CUDA out of memory")
    api._state.engine.iterate = boom
    with pytest.raises(RuntimeError, match="out of memory"):
        api.do_run(args)
    assert "Try reducing --num-cuts" in capsys.readouterr().out     # pixray.py:1625-1628


def test_vdiff_loop_renoises_and_restarts_adam(fake, tmp_path):
    sd = {"dummy": torch.zeros(1)}
    args = _init(tmp_path, prompts="x", drawer="vdiff", clip_models="ViT-B/16", iterations=6, learning_rate_drops=None,
                 b200_weights={"vdiff": sd})
    eng = api._state.engine
    assert "vdiff_set_schedule" in eng.names() and "vdiff_set_clip_embed" in eng.names()
    assert api.do_run(args) is True
    renoise = [c[1]["i"] for c in eng.calls if c[0] == "vdiff_renoise"]
    assert renoise == [1, 2, 3, 4, 5, 6]                              # every step from the second on (pixray.py:1489-1495)
    lrs = [c[1]["lr"] for c in eng.calls if c[0] == "iterate"]
    d = api._state.drawer
    assert lrs[0] == pytest.approx(0.2)
    for it in range(2, 6):                                            # lr of iteration it was set after iteration it-1
        assert lrs[it] == pytest.approx(min(float(d.sigmas[it - 1] / d.alphas[it - 1]) * 0.001, 0.01))


def test_custom_losses_and_image_prompts_reach_the_engine(fake, tmp_path):
    target = torch.rand(1, 3, 32, 32)
    args = _init(tmp_path, prompts="x", clip_models="ViT-B/16", iterations=3, custom_loss="smoothness:0.5,symmetry",
                 image_prompts=[target], image_prompt_weight=0.7)
    eng = api._state.engine
    assert [a[0] for a in eng.aux] == [E.LOSS_SMOOTHNESS, E.LOSS_SYMMETRY] and eng.aux[0][1] == 0.5 and eng.aux[1][1] == 1
    imgs, w = eng.image_prompts
    # the target keeps ITS size (resize_image never forces the canvas size, pixray.py:514-518; MakeCutouts pools any size)
    assert len(imgs) == 1 and tuple(imgs[0].shape) == (1, 3, 32, 32) and w == [0.7]
    assert api._state.loss_buf.size == eng.num_losses() == 2 + 1 + 2  # text + vector, image prompt, two custom losses
    assert api.do_run(args) is True


def test_run_is_the_one_stop_call(fake, tmp_path):
    (tmp_path / "vectors").mkdir(exist_ok=True)
    (tmp_path / "vectors" / "textoff.json").write_text(json.dumps({"ViT-B/16": [[0.1] * 512]}))
    os.environ["PIXRAY_ROOT"] = str(tmp_path)
    api.run("a cat", "fast_pixel", size=[32, 32], pixel_size=[8, 8], clip_models="ViT-B/16", iterations=4, num_cuts=4,
            outdir="", b200_allow_synthetic=True)
    assert [c[1]["it"] for c in api._state.engine.calls if c[0] == "iterate"] == [0, 1, 2, 3]
    assert isinstance(api._state.drawer, P.FastPixelDrawer) and tuple(api._state.drawer.get_z().shape) == (1, 3, 8, 8)


def test_plugin_train_iteration_call_sequence(fake, tmp_path):
    """The per-op plugin path (what a pixray loop written against the plugin objects executes): one iteration issues the
    reference's sequence, and Prompt.forward does not hand the engine's own embeddings back in (the engine keeps them
    un-normalised for its backward)."""
    _init(tmp_path, prompts="a|b", clip_models="ViT-B/16", iterations=3)
    st = api._state
    eng = st.engine
    eng.calls.clear()
    opt = P.Optimizer(st.session, st.drawer, 0.05)
    st.session.begin_iteration(0, fill=0.5)
    losses = P.train_iteration(st.session, st.drawer, st.make_cutouts, st.perceptors, st.prompt_tables, opt)
    assert len(losses) == 3
    assert eng.names() == ["reset_optimizer", "synth", "make_cutouts", "encode_image", "prompt_loss", "prompt_loss",
                           "prompt_loss", "backward", "set_z_grad", "step"]
    assert not any(c[1]["passed_embeds"] for c in eng.calls if c[0] == "prompt_loss")
    mc = [c for c in eng.calls if c[0] == "make_cutouts"][0][1]
    assert mc["transforms"] == "ndarray" and mc["color_jitter"] == "ndarray" and mc["noise"] == "Tensor"
    assert st.make_cutouts.transforms is None                        # per-iteration cache cleared (pixray.py:1339-1342)
    assert torch.equal(st.drawer.get_z().grad, torch.ones(eng.z_shape))
    step = [c for c in eng.calls if c[0] == "step"][0][1]
    assert step["lr"] == 0.05 and step["it"] == 0


def test_package_exposes_the_reference_entry_points():
    import pixray_b200 as pixray
    for name in ("run", "reset_settings", "add_settings", "get_settings", "apply_settings", "do_init", "do_run",
                 "add_custom_loss"):
        assert callable(getattr(pixray, name)), name
    with pytest.raises(AttributeError):
        pixray.no_such_thing


def test_pixel_drawer_grid_follows_the_reference_defaults(fake, tmp_path):
    """fast_pixeldrawer.py:37-63: 40x40 on a square canvas when no pixel_size is given, pixel_scale divides the grid, and the
    grid never exceeds the canvas."""
    assert P.FastPixelDrawer.grid_for((256, 256)) == (40, 40)
    assert P.FastPixelDrawer.grid_for((192, 108)) == (45, 80)
    assert P.FastPixelDrawer.grid_for((128, 160)) == (50, 40)
    assert P.FastPixelDrawer.grid_for((256, 256), pixel_scale=2.0) == (20, 20)
    assert P.FastPixelDrawer.grid_for((256, 256), pixel_size=[64, 32]) == (32, 64)
    assert P.FastPixelDrawer.grid_for((32, 32), verbose=False) == (32, 32)
    args = _init(tmp_path, prompts="x", drawer="fast_pixel", clip_models="ViT-B/32", size=[256, 256])
    assert api._state.engine.kw["grid"] == (40, 40) and tuple(api._state.drawer.get_z().shape) == (1, 3, 40, 40)
    api.reset_settings()
    args = _init(tmp_path, prompts="x", drawer="fast_pixel", clip_models="ViT-B/32", size=[256, 256], pixel_scale=0.5)
    assert api._state.engine.kw["grid"] == (80, 80)


def test_aesthetic_loss_is_usable_through_the_settings(fake, tmp_path):
    """custom_loss='aesthetic' (pixray.py:131-140, Losses/AestheticLoss.py): the linear AVA head the reference downloads comes
    in through `aesthetic_head` (dict or .pth path); without it the error names the missing file."""
    head = {"weight": torch.linspace(-1, 1, 512).reshape(1, 512), "bias": torch.tensor([0.25])}
    path = tmp_path / "ava_head.pth"
    torch.save(head, path)
    for spec in (head, str(path)):
        api.reset_settings()
        _init(tmp_path, prompts="x", clip_models="ViT-B/16", custom_loss="aesthetic:0.5", aesthetic_target=7, aesthetic_head=spec)
        kind, weight, params = api._state.engine.aux[-1]
        assert kind == E.LOSS_AESTHETIC and weight == 0.5
        assert params[0] == 7 and abs(params[1] - 0.25) < 1e-7 and len(params) == 2 + 512 and abs(params[2] + 1.0) < 1e-6
    api.reset_settings()
    with pytest.raises(FileNotFoundError):
        _init(tmp_path, prompts="x", clip_models="ViT-B/16", custom_loss="aesthetic")


def test_file_image_prompts_keep_their_aspect_ratio(fake, tmp_path):
    """resize_image (pixray.py:514-518): area = min(source area, canvas area), the source's aspect ratio is kept."""
    from PIL import Image
    wide = tmp_path / "wide.png"
    Image.fromarray((np.random.default_rng(0).random((40, 160, 3)) * 255).astype(np.uint8)).save(wide)
    big = tmp_path / "big.png"
    Image.fromarray((np.random.default_rng(1).random((300, 200, 3)) * 255).astype(np.uint8)).save(big)
    _init(tmp_path, prompts="x", clip_models="ViT-B/16", size=[64, 64], image_prompts=[str(wide), str(big)])
    imgs, _ = api._state.engine.image_prompts
    # 160x40 (area 6400 > 64*64 = 4096): ratio 4 -> 128 x 32;  200x300: ratio 2/3 -> 52 x 78
    assert tuple(imgs[0].shape[-2:]) == (32, 128) and tuple(imgs[1].shape[-2:]) == (78, 52)
    assert 0.0 <= float(imgs[0].min()) and float(imgs[0].max()) <= 1.0


def test_spot_prompts_reach_the_engine(fake, tmp_path):
    """args.spot_prompts / spot_prompts_off (pixray.py:917-931) with the reference's own mask image (inputs/spot_square.png,
    stored as tests/golden/spot_square.png; fetch_spot_indexes pixray.py:370-394) resized to the cut size."""
    (tmp_path / "inputs").mkdir(exist_ok=True)
    import shutil
    shutil.copy(os.path.join(os.path.dirname(__file__), "golden", "spot_square.png"), tmp_path / "inputs" / "spot_square.png")
    _init(tmp_path, prompts="x", clip_models="ViT-B/32,ViT-B/16", spot_prompts="a red circle:2|a dot", spot_prompts_off="the sky")
    eng = api._state.engine
    calls = [c for c in eng.calls if c[0] == "set_spot_prompts"]
    assert [(c[1]["clip"], c[1]["which"], c[1]["n"]) for c in calls] == [(0, 1, 2), (0, 0, 1), (1, 1, 2), (1, 0, 1)]
    assert eng.spot_mask.shape == (3, 224, 224) and 0.05 < eng.spot_mask.mean() < 0.95
    api.reset_settings()
    with pytest.raises(FileNotFoundError):
        os.environ["PIXRAY_ROOT"] = str(tmp_path / "nowhere")
        _init2 = dict(size=[64, 64], num_cuts=8, outdir="", seed="7", b200_allow_synthetic=True, prompts="x", clip_models="ViT-B/16",
                      spot_prompts="a dot", vector_prompts="none")
        api.add_settings(**_init2)
        cwd = os.getcwd()
        os.chdir(tmp_path / "vectors")
        try:
            api.do_init(api.apply_settings())
        finally:
            os.chdir(cwd)


def test_default_start_is_an_encoded_noise_image_and_overlays_re_encode(fake, tmp_path):
    """pixray.py:674-727: init_noise='pixels' (default) -> a fractal-noise image in [-1, 1] through drawer.init_from_tensor
    (model.encode on the engine); init_image replaces it; overlays paste + re-encode every overlay_every iterations
    (re_average_z, pixray.py:1408-1420)."""
    from PIL import Image
    _init(tmp_path, prompts="x", clip_models="ViT-B/16")
    enc = [c for c in api._state.engine.calls if c[0] == "vqgan_encode"]
    assert len(enc) == 1 and enc[0][1]["shape"] == (1, 3, 64, 64) and -1.0 <= enc[0][1]["lo"] < -0.5 and 0.5 < enc[0][1]["hi"] <= 1.0
    api.reset_settings()
    _init(tmp_path, prompts="x", clip_models="ViT-B/16", init_noise="none")
    assert not [c for c in api._state.engine.calls if c[0] == "vqgan_encode"]      # legacy start: random codebook rows
    init = tmp_path / "init.png"
    Image.fromarray(np.full((40, 50, 3), 200, np.uint8)).save(init)
    ov = tmp_path / "ov.png"
    Image.fromarray(np.dstack([np.zeros((64, 64, 3), np.uint8), np.full((64, 64), 255, np.uint8)]), mode="RGBA").save(ov)
    api.reset_settings()
    args = _init(tmp_path, prompts="x", clip_models="ViT-B/16", init_image=str(init), overlay_image=str(ov), overlay_every=3,
                 overlay_alpha=128, iterations=7)
    enc = [c for c in api._state.engine.calls if c[0] == "vqgan_encode"]
    assert len(enc) == 1 and abs(enc[0][1]["lo"] - (200 / 255 * 2 - 1)) < 1e-6 and enc[0][1]["lo"] == enc[0][1]["hi"]
    assert api.do_run(args) is True
    names = api._state.engine.names()
    # iterations 0, 3 and 6 render (synth), paste the overlay and re-encode before their step
    assert names.count("vqgan_encode") == 1 + 3
    first = names.index("iterate")
    assert names[first - 2:first] == ["synth", "vqgan_encode"]


def test_filters_reach_the_engine(fake, tmp_path):
    """args.filters = "name:weight,..." (pixray.py:651-668) with the filters' own settings (filters/wallpaper.py:17-20,
    filters/colorlookup.py:32-35); unknown names raise like the reference."""
    _init(tmp_path, prompts="x", clip_models="ViT-B/16", filters="wallpaper:0.5,lookup,tiler", wallpaper_type="horizontal",
          wallpaper_edge_match=8, lookup_beta=4.0, palette="#ff0000;#00ff00")
    f = api._state.engine.filters
    assert [(k, w) for k, w, _ in f] == [(E.FILTER_WALLPAPER, 0.5), (E.FILTER_LOOKUP, 1), (E.FILTER_TILER, 1)]
    assert f[0][2] == [2, 8] and f[1][2] == [4.0, 1.0, 0.0, 0.0, 0.0, 1.0, 0.0] and f[2][2] == []
    assert api._state.loss_buf.size == 3 + 2
    api.reset_settings()
    api.add_settings(prompts="x", filters="sepia")
    with pytest.raises(ValueError):
        api.apply_settings()
    api.reset_settings()
    _init(tmp_path, prompts="x", clip_models="ViT-B/16", filters="lookup")          # built-in 16-colour table
    assert len(api._state.engine.filters[0][2]) == 1 + 16 * 3


def test_init_weight_family_and_image_labels_become_anchors(fake, tmp_path):
    """pixray.py:833-850, 1344-1375: image_labels first, then init_weight (spherical), init_weight_dist (mse),
    init_weight_pix (l1 on the image), init_weight_cos -- anchored on z_orig = the encoded init image (pixray.py:719)."""
    from PIL import Image
    init = tmp_path / "init.png"
    Image.fromarray(np.full((64, 64, 3), 100, np.uint8)).save(init)
    for k in range(2):
        Image.fromarray(np.full((32, 48, 3), 50 + 100 * k, np.uint8)).save(tmp_path / f"label{k}.png")
    _init(tmp_path, prompts="x", clip_models="ViT-B/16", init_image=str(init), init_weight=0.5, init_weight_dist=0.25,
          init_weight_pix=2.0, init_weight_cos=0.125, image_labels=str(tmp_path / "label*.png"), image_label_weight=3.0)
    eng = api._state.engine
    assert [(k, w) for k, w, _ in eng.anchors] == [(E.ANCHOR_SPHERICAL, 3.0), (E.ANCHOR_SPHERICAL, 0.5), (E.ANCHOR_MSE, 0.25),
                                                   (E.ANCHOR_PIX, 2.0), (E.ANCHOR_COS, 0.125)]
    assert eng.anchors[3][2].shape == (1, 3, 64, 64) and abs(float(eng.anchors[3][2].max()) - 100 / 255) < 1e-6
    assert eng.names().count("vqgan_encode") == 1 + 2            # the init image and the two label images
    assert api._state.loss_buf.size == 2 + 5
    api.reset_settings()
    with pytest.raises(ValueError, match="init_image"):          # the reference dereferences z_orig = None there
        _init(tmp_path, prompts="x", clip_models="ViT-B/16", init_weight=0.5)
