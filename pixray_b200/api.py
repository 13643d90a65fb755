"""pixray's module-level entry points on the B200 engine: `run`, `reset_settings`, `add_settings`, `get_settings`,
`apply_settings`, `do_init`, `do_run`, `add_custom_loss` (pixray.py:2005-2124) -- the five calls the reference's
front-ends use (run.py, cogrun.py) plus the notebook one-liner.

Scope (SURVEY.md 8): the per-iteration hot path.  Every option of the reference's parser is KNOWN here (same dest,
same default: the "requested setting not found" check of pixray.py:2088-2093 behaves identically), but options that
switch on something outside the hot path (spot prompts, overlays, animation, init images through the VQGAN encoder,
filters, transparency, the AdamP optimiser, SLIP perceptors, video) raise NotImplementedError when they are set to a
non-default value instead of being silently ignored.  `optimiser` takes Adam, AdamW, Adagrad, Adamax or DiffGrad, each
with its library's defaults like the reference builds them (pixray.py:536-553).  What the reference fetches from the network at init time comes in
through three extra settings instead:

    b200_weights        {"vqgan": state_dict | path, "ViT-B/16": state_dict | path, ...} with the reference's own keys
                        (taming `state_dict`, openai-CLIP `visual.*`); None = seeded synthetic weights (benchmarks)
    b200_text_encoder   callable(clip_model_name, text) -> [1, D] tensor (e.g. the reference's perceptor.encode_text);
                        the text towers are init-time and stay in PyTorch
    b200_allow_synthetic  accept seeded pseudo-embeddings for text prompts when no encoder is given (default False)

One session per process, like the reference's module globals (pixray.py:1022-1063)."""
import argparse
import hashlib
import json
import os
import random
import zlib
from types import SimpleNamespace

import numpy as np
import torch

from . import engine as E
from . import filters as FL
from . import losses as L
from . import plugins as P
from . import synthetic as S
from .util import apply_overlay, get_learning_rate_drops, parse_unit, split_pipes

# pixray.class_table (pixray.py:74-113) restricted to the drawers of the BASELINE configs; "pixel" is the rect grid the
# reference renders through diffvg, which fast_pixel reproduces (SURVEY.md 2, row 6)
class_table = {"vqgan": P.VqganDrawer, "fast_pixel": P.FastPixelDrawer, "pixel": P.FastPixelDrawer, "fft": P.FftDrawer,
               "vdiff": P.VdiffDrawer}
_DRAWER_KIND = {"vqgan": E.DRAWER_VQGAN, "fast_pixel": E.DRAWER_PIXEL, "pixel": E.DRAWER_PIXEL, "fft": E.DRAWER_FFT,
                "vdiff": E.DRAWER_VDIFF}
loss_class_table = L.loss_class_table
filters_class_table = FL.filters_class_table

global_pixray_settings = {}
_engine_factory = E.B200Engine  # tests substitute a recording stand-in; the product has no other implementation


def str2bool(v):
    if isinstance(v, bool):
        return v
    if v.lower() in ("yes", "true", "t", "y", "1"):
        return True
    if v.lower() in ("no", "false", "f", "n", "0"):
        return False
    raise argparse.ArgumentTypeError("Boolean value expected.")


# (flags, dest, type, default[, nargs]) -- setup_parser, pixray.py:1722-1822
_OPTIONS = [
    (("-p", "--prompts"), "prompts", str, []), (("-sp", "--spot"), "spot_prompts", str, []),
    (("-spo", "--spot_off"), "spot_prompts_off", str, []), (("-spf", "--spot_file"), "spot_file", str, None),
    (("-l", "--labels"), "labels", str, []), (("-vp", "--vector_prompts"), "vector_prompts", str, "textoff"),
    (("-ip", "--image_prompts"), "image_prompts", str, []),
    (("-ipw", "--image_prompt_weight"), "image_prompt_weight", float, None),
    (("-ips", "--image_prompt_shuffle"), "image_prompt_shuffle", str2bool, False),
    (("-il", "--image_labels"), "image_labels", str, None), (("-ilw", "--image_label_weight"), "image_label_weight", float, 1.0),
    (("-i", "--iterations"), "iterations", int, None), (("-se", "--save_every"), "save_every", str, 10),
    (("-si", "--save_intermediates"), "save_intermediates", str2bool, True),
    (("-de", "--display_every"), "display_every", str, 20), (("-dc", "--display_clear"), "display_clear", str2bool, False),
    (("-ove", "--overlay_every"), "overlay_every", str, "10 iterations"),
    (("-ovo", "--overlay_offset"), "overlay_offset", str, "0 iterations"),
    (("-ovu", "--overlay_until"), "overlay_until", str, None), (("-ovi", "--overlay_image"), "overlay_image", str, None),
    (("--quality",), "quality", str, "normal"), (("-asp", "--aspect"), "aspect", str, "widescreen"),
    (("-ezs", "--ezsize"), "ezsize", str, None), (("-sca", "--scale"), "scale", float, None),
    (("-ova", "--overlay_alpha"), "overlay_alpha", int, None), (("-s", "--size"), "size", int, None, 2),
    (("-ii", "--init_image"), "init_image", str, None), (("-iia", "--init_image_alpha"), "init_image_alpha", int, 200),
    (("-in", "--init_noise"), "init_noise", str, "pixels"), (("-ti", "--target_images"), "target_images", str, None),
    (("-anim", "--animation_dir"), "animation_dir", str, None), (("-ana", "--animation_alpha"), "animation_alpha", int, 128),
    (("-iw", "--init_weight"), "init_weight", float, None), (("-iwd", "--init_weight_dist"), "init_weight_dist", float, 0.0),
    (("-iwc", "--init_weight_cos"), "init_weight_cos", float, 0.0), (("-iwp", "--init_weight_pix"), "init_weight_pix", float, 0.0),
    (("--perceptors",), "perceptors", str, "clip"), (("--clip_models",), "clip_models", str, None),
    (("-nps", "--noise_prompt_seeds"), "noise_prompt_seeds", int, [], "*"),
    (("-npw", "--noise_prompt_weights"), "noise_prompt_weights", float, [], "*"),
    (("-lr", "--learning_rate"), "learning_rate", float, 0.2),
    (("-lrd", "--learning_rate_drops"), "learning_rate_drops", str, [75], "*"),
    (("-as", "--auto_stop"), "auto_stop", str2bool, False), (("-cuts", "--num_cuts"), "num_cuts", int, None),
    (("-bats", "--batches"), "batches", int, None), (("-cutp", "--cut_power"), "cut_pow", float, 1.0),
    (("--seed",), "seed", str, None), (("-opt", "--optimiser"), "optimiser", str, "Adam"),
    (("-vid", "--video"), "make_video", str2bool, False), (("-d", "--deterministic"), "cudnn_determinism", str2bool, False),
    (("-cud", "--cuda_device"), "cuda_device", str, "cuda:0"), (("--palette",), "palette", str, None),
    (("--transparent",), "transparent", str2bool, False), (("--transparent_weight",), "transparent_weight", float, 0.0),
    (("--alpha_use_g",), "alpha_use_g", str2bool, False), (("--alpha_gamma",), "alpha_gamma", float, 4.0),
    (("--output",), "output", str, "output.png"), (("--outdir",), "outdir", str, "outputs/%DATE%_%SEQ%"),
]
_ENGINE_OPTIONS = [(("--b200_weights",), "b200_weights", None, None), (("--b200_text_encoder",), "b200_text_encoder", None, None),
                   (("--b200_allow_synthetic",), "b200_allow_synthetic", str2bool, False),
                   # checkdrop / learning-rate drops / auto-stop decided on the device, no per-iteration host sync
                   # (pxr_set_schedule); False keeps the reference's host-side control flow (one loss readback per iteration)
                   (("--b200_device_checkdrop",), "b200_device_checkdrop", str2bool, True),
                   # cutout-sharded multi-GPU run (one process per GPU, torch.distributed already initialised by the
                   # launcher): this process is rank b200_rank of b200_world and drives cuda:<LOCAL_RANK>
                   (("--b200_rank",), "b200_rank", int, 0), (("--b200_world",), "b200_world", int, 1)]

# options that leave the hot path: dest -> the value(s) that keep them off
_OFF_PATH = {
    "labels": ([],),
    "target_images": (None, []), "animation_dir": (None,),
    "perceptors": ("clip",), "optimiser": tuple(E.OPTIMISERS), "make_video": (False,), "transparent": (False,),
    "image_prompt_shuffle": (False,),
}

quality_to_clip_models_table = {"draft": "ViT-B/16", "normal": "ViT-B/32,ViT-B/16", "better": "RN50,ViT-B/32,ViT-B/16",
                                "best": "RN50x4,ViT-B/32,ViT-B/16", "supreme": "RN50x4,RN101,ViT-B/32,ViT-B/16"}
quality_to_iterations_table = {"draft": 200, "normal": 250, "better": 300, "best": 350, "supreme": 400}
quality_to_scale_table = {"draft": 1, "normal": 2, "better": 3, "best": 4, "supreme": 5}
quality_to_num_cuts_table = {"draft": 24, "normal": 30, "better": 36, "best": 12, "supreme": 8}
quality_to_batches_table = {"draft": 1, "normal": 1, "better": 1, "best": 2, "supreme": 4}
size_to_scale_table = {"small": 1, "medium": 2, "large": 4}
aspect_to_size_table = {"square": [144, 144], "portrait": [128, 160], "widescreen": [192, 108]}


# ------------------------------------------------------------------------------------------------ settings
def reset_settings():
    global global_pixray_settings
    global_pixray_settings = {}


def add_settings(**kwargs):
    for k, v in kwargs.items():
        global_pixray_settings[k] = v


def get_settings():
    return global_pixray_settings.copy()


def add_custom_loss(name, customloss):
    """pixray.py:2104-2109."""
    assert issubclass(customloss, L.LossInterface)
    loss_class_table.update({name: customloss})


def setup_parser(vq_parser):
    for spec in _OPTIONS + _ENGINE_OPTIONS:
        flags, dest, typ, default = spec[:4]
        kw = dict(dest=dest, default=default)
        if typ is not None:
            kw["type"] = typ
        if len(spec) > 4:
            kw["nargs"] = spec[4]
        vq_parser.add_argument(*flags, **kw)
    return vq_parser


def _spec_names(spec):
    return [chunk.strip().split(":")[0].split("->")[0] for chunk in spec.split(",")]


def apply_settings():
    """Two-pass parse like pixray.py:2055-2102: drawer / filters / losses first (they contribute options), then the
    rest; unknown keys of the settings dict raise ValueError.  Library use only: sys.argv is never read."""
    first = argparse.ArgumentParser(description="Image generation using VQGAN+CLIP")
    first.add_argument("--drawer", type=str, default="vqgan", dest="drawer")
    first.add_argument("--filters", type=str, default=None, dest="filters")
    first.add_argument("--losses", "--custom_loss", type=str, default=None, dest="custom_loss")
    core, _ = first.parse_known_args(args=[], namespace=SimpleNamespace(**global_pixray_settings))
    if core.drawer not in class_table:
        raise ValueError(f"drawer '{core.drawer}' is not on the hot-path scope; available: {sorted(class_table)}")
    vq_parser = setup_parser(first)
    class_table[core.drawer].add_settings(vq_parser)
    if core.filters is not None:  # pixray.py:2072-2078
        for name in _spec_names(core.filters):
            if name not in filters_class_table:
                raise ValueError(f"Requested filter not found, aborting: {name}")
            filters_class_table[name].add_settings(vq_parser)
    if core.custom_loss is not None:
        for name in _spec_names(core.custom_loss):
            if name not in loss_class_table:
                raise ValueError(f"Requested loss not found, aborting: {name}")
            loss_class_table[name].add_settings(vq_parser)
    dests = [a.dest for a in vq_parser._actions]
    for k in global_pixray_settings:
        if k not in dests and k != "skip_args":
            raise ValueError(f"Requested setting not found, aborting: {k}={global_pixray_settings[k]}")
    return process_args(vq_parser, SimpleNamespace(**global_pixray_settings))


def _parse_palette(p):
    if p is None or not isinstance(p, str):
        return p
    cols = []
    for chunk in p.replace("\\", "").split(";"):
        c = chunk.strip().lstrip("#")
        if len(c) != 6:
            raise NotImplementedError("palette: pass a list of [r, g, b] in [0, 1] or '#rrggbb;#rrggbb;...' "
                                      "(named / gradient palettes need matplotlib's colour tables)")
        cols.append([int(c[i:i + 2], 16) / 255.0 for i in (0, 2, 4)])
    return cols


def process_args(vq_parser, namespace):
    """pixray.py:1824-1997 for the hot-path options: quality presets, size, unit strings, prompt splitting."""
    args = vq_parser.parse_args(args=[], namespace=namespace)
    for dest, off in _OFF_PATH.items():
        if getattr(args, dest, off[0]) not in off:
            raise NotImplementedError(f"setting '{dest}' leaves the per-iteration hot path this engine covers (SURVEY.md 8)")
    if args.quality not in quality_to_clip_models_table:
        raise ValueError(f"Quality setting not understood, aborting -> {args.quality}")
    if args.clip_models is None:
        args.clip_models = quality_to_clip_models_table[args.quality]
    if args.iterations is None:
        args.iterations = quality_to_iterations_table[args.quality]
    if args.num_cuts is None:
        args.num_cuts = quality_to_num_cuts_table[args.quality]
    if args.batches is None:
        args.batches = quality_to_batches_table[args.quality]
    if args.ezsize is None and args.scale is None:
        args.scale = quality_to_scale_table[args.quality]
    if args.size is None:
        size_scale = args.scale
        if size_scale is None:
            if args.ezsize not in size_to_scale_table:
                raise ValueError(f"EZ Size not understood, aborting -> {args.ezsize}")
            size_scale = size_to_scale_table[args.ezsize]
        if args.aspect not in aspect_to_size_table:
            raise ValueError(f"aspect not understood, aborting -> {args.aspect}")
        base = aspect_to_size_table[args.aspect]
        args.size = [int(size_scale * base[0]), int(size_scale * base[1])]
    if isinstance(args.init_noise, str) and args.init_noise.lower() == "none":
        args.init_noise = None
    args.prompts = split_pipes(args.prompts)
    args.save_every = parse_unit(args.save_every, args.iterations, "save_every", "i")
    args.display_every = parse_unit(args.display_every, args.iterations, "display_every", "i")
    args.overlay_offset = parse_unit(args.overlay_offset, args.iterations, "overlay_offset", "i")
    args.overlay_until = parse_unit(args.overlay_until, args.iterations, "overlay_until", "i")
    args.overlay_every = parse_unit(args.overlay_every, args.iterations, "overlay_every", "i")
    if args.image_prompts and isinstance(args.image_prompts, str):
        args.image_prompts = [args.image_prompts]
    if args.vector_prompts:
        if args.vector_prompts.lower() == "none" or args.vector_prompts == "0":
            args.vector_prompts = []
        else:
            args.vector_prompts = [phrase.strip() for phrase in args.vector_prompts.split("|")]
    else:
        args.vector_prompts = []
    args.palette = _parse_palette(args.palette)
    args.clip_models = [m.strip() for m in args.clip_models.split(",")]
    args.learning_rate_drops = get_learning_rate_drops(args.learning_rate_drops, args.iterations)
    return args


# ------------------------------------------------------------------------------------------------ session state
_state = SimpleNamespace(engine=None, session=None, drawer=None, perceptors=[], make_cutouts=None, lr=0.0,
                         cur_iteration=0, best_loss=1e20, best_iter=0, num_loss_drop=0, max_loss_drops=0,
                         iter_drop_delay=12, losses=None, loss_buf=None, seed=None, custom=[], managed=False, stop_iter=None)


def _seed_everything(args):
    """pixray.py:588-606."""
    if args.seed is None:
        seed = torch.seed()
    else:
        seed = int.from_bytes(hashlib.sha512(str(args.seed).encode()).digest(), "big") % 0x100000000
    int_seed = int(seed) % (2 ** 30)
    torch.manual_seed(seed)
    np.random.seed(int_seed)
    random.seed(int_seed)
    return int_seed


def _load_state_dict(spec):
    if isinstance(spec, (str, os.PathLike)):
        try:
            obj = torch.jit.load(str(spec), map_location="cpu").state_dict()  # openai-CLIP ships TorchScript archives
        except Exception:
            obj = torch.load(str(spec), map_location="cpu", weights_only=False)
        if isinstance(obj, dict) and "state_dict" in obj:  # taming checkpoints (vqgan.py:128-133)
            obj = obj["state_dict"]
        return obj
    return spec


def _vector_table(name):
    """`vectors/<name>.json` next to the reference checkout (pixray.py:893-901)."""
    if "json" in name:
        cands = [name]
    else:
        cands = [f"vectors/{name}.json", f"pixray/vectors/{name}.json"]
        if os.environ.get("PIXRAY_ROOT"):
            cands.append(os.path.join(os.environ["PIXRAY_ROOT"], "vectors", f"{name}.json"))
    for c in cands:
        if os.path.exists(c):
            with open(c) as f:
                return json.load(f)
    raise FileNotFoundError(f"vector prompt file not found (tried {cands}); set PIXRAY_ROOT or vector_prompts='none'")


def _text_embed(args, clip_model, txt, out_dim):
    if args.b200_text_encoder is not None:
        return torch.as_tensor(args.b200_text_encoder(clip_model, txt), dtype=torch.float32).reshape(1, out_dim).cpu()
    if not args.b200_allow_synthetic:
        raise ValueError("text prompts need a text tower: pass b200_text_encoder=callable(clip_model, text) -> [1, D] "
                         "(e.g. the reference's perceptor.encode_text), or b200_allow_synthetic=True for seeded "
                         "pseudo-embeddings")
    gen = torch.Generator().manual_seed(zlib.crc32(f"{clip_model}|{txt}".encode()))
    return torch.empty([1, out_dim]).normal_(generator=gen)  # the reference's own noise-prompt recipe, pixray.py:955-958


def _side(args, num_resolutions):
    if num_resolutions is not None:  # pixray.py:619-624
        f = 2 ** (num_resolutions - 1)
        return (args.size[0] // f) * f, (args.size[1] // f) * f
    return args.size[0], args.size[1]


def do_init(args):
    """pixray.py:569-1020 for the hot path: engine + drawer + perceptors + cutouts + prompts + losses + optimiser."""
    st = _state
    for m in args.clip_models:
        if m not in E.CLIP_ARCH:
            raise NotImplementedError(f"perceptor '{m}': only the ViT image towers {sorted(E.CLIP_ARCH)} are built")
    if len(args.clip_models) > 2:
        raise NotImplementedError("at most two perceptors per session")
    st.seed = _seed_everything(args)
    kind = _DRAWER_KIND[args.drawer]
    n_levels = len(E.VQGAN_F16_16384["ch_mult"]) if kind == E.DRAWER_VQGAN else None
    sideX, sideY = _side(args, n_levels)
    # global_aspect_width = args.size[0] / args.size[1] (pixray.py:1931: the REQUESTED size, before the drawer rounds it):
    # != 1 stretches the pooled image before the warps and changes the wide augmentation stack (pixray.py:420-432, 468-472)
    aspect = float(args.size[0]) / float(args.size[1])
    device = int(str(args.cuda_device).split(":")[1]) if ":" in str(args.cuda_device) else 0
    clip_cfgs = [E.CLIP_ARCH[m] for m in args.clip_models]
    kw = dict(drawer=kind, image_hw=(sideY, sideX), cutn=args.num_cuts, clip=clip_cfgs, seed=st.seed, device=device)
    if aspect != 1.0:
        kw["cut_aspect"] = aspect
    world = int(getattr(args, "b200_world", 1) or 1)
    if world > 1:
        kw.update(rank=int(args.b200_rank), world=world)
    if kind == E.DRAWER_PIXEL:  # fast_pixeldrawer.py:37-63: 40x40 / 40x50 / 80x45 default grid, pixel_scale, clamp to canvas
        kw["grid"] = P.FastPixelDrawer.grid_for((sideX, sideY), getattr(args, "pixel_size", None), getattr(args, "pixel_scale", None))
        print(f"Running fast pixeldrawer with {kw['grid'][1]}x{kw['grid'][0]} grid")
    if kind == E.DRAWER_FFT:
        kw.update(fft_decay=args.fft_decay, fft_colors=args.fft_colors)
    eng = _engine_factory(**kw)
    weights = args.b200_weights or {}
    if kind in (E.DRAWER_VQGAN, E.DRAWER_VDIFF):
        key = "vqgan" if kind == E.DRAWER_VQGAN else "vdiff"
        if key in weights:
            vq_sd = _load_state_dict(weights[key])
        elif kind == E.DRAWER_VQGAN:
            vq_sd = S.vqgan_state_dict(E.VQGAN_F16_16384, 0, with_encoder=True)
        elif args.b200_allow_synthetic:
            vq_sd = S.vdiff_state_dict(0)
        else:
            raise ValueError("the vdiff drawer needs b200_weights['vdiff'] (the cc12m_1 checkpoint's state_dict), or "
                             "b200_allow_synthetic=True for seeded random weights")
        eng.load_module(E.MOD_VQGAN, vq_sd)
    for i, m in enumerate(args.clip_models):
        sd = _load_state_dict(weights[m]) if m in weights else S.clip_state_dict(E.CLIP_ARCH[m], 1 + i)
        eng.load_module(E.MOD_CLIP0 + i, sd)
    eng.finalize()
    if world > 1:
        eng.init_comm()
    st.engine, st.session = eng, P.Session(eng)
    drawer = class_table[args.drawer](args, st.session)
    drawer.load_model(args, eng.device)
    # ---- image initialisation (pixray.py:674-727): a noise / gradient / blank start image, optionally an init image, into
    # drawer.init_from_tensor(t * 2 - 1) -- for the VQGAN drawer that is model.encode on the engine (pxr_vqgan_encode)
    st.init_image_tensor, st.z_orig = None, None
    if kind in (E.DRAWER_VQGAN, E.DRAWER_PIXEL) and (args.init_image or args.init_noise):
        from PIL import Image
        from .util import random_gradient_image, random_noise_image
        rng = np.random.default_rng(st.seed)
        w0, h0 = args.size[0], args.size[1]
        if args.init_noise == "pixels":
            img = Image.fromarray(random_noise_image(w0, h0, rng))
        elif args.init_noise == "gradient":
            img = Image.fromarray(random_gradient_image(w0, h0, rng))
        elif args.init_noise == "snow":
            img = Image.fromarray(rng.integers(0, 255, (w0, h0, 3), dtype=np.uint8))  # old_random_noise_image: (w, h, 3)
        else:
            img = Image.new(mode="RGB", size=(w0, h0), color=(255, 255, 255))
        starting_image = img.convert("RGB").resize((sideX, sideY), Image.LANCZOS)
        to_t = lambda im: torch.from_numpy(np.asarray(im, dtype=np.float32) / 255.0).permute(2, 0, 1).unsqueeze(0)  # noqa: E731
        if args.init_image:
            init_rgb = Image.open(args.init_image).convert("RGB").resize((sideX, sideY), Image.LANCZOS)
            st.init_image_tensor = to_t(init_rgb)
            drawer.init_from_tensor(st.init_image_tensor * 2 - 1)  # the init image itself, not the alpha paste (pixray.py:715-716)
            st.z_orig = drawer.get_z_copy()                        # pixray.py:719
        else:
            drawer.init_from_tensor(to_t(starting_image) * 2 - 1)
    elif kind == E.DRAWER_VQGAN:
        # init_image and init_noise both off: the legacy start (VqganDrawer.rand_init, vqgan.py:162-171): random codebook rows
        code = torch.as_tensor(vq_sd["quantize.embedding.weight"], dtype=torch.float32)
        idx = torch.randint(code.shape[0], (eng.z_shape[2] * eng.z_shape[3],))
        drawer.set_z(code[idx].T.reshape(eng.z_shape))
    elif kind == E.DRAWER_PIXEL:
        drawer.init_from_tensor(torch.rand(1, 3, sideY, sideX) * 2 - 1)
    else:
        drawer.init_from_tensor(None)
    # overlays (pixray.py:729-745, 1408-1420): one RGBA image pasted over the current image every overlay_every iterations
    st.overlay_rgba = None
    if args.overlay_image is not None:
        from PIL import Image
        ov = Image.open(args.overlay_image).convert("RGBA").resize((sideX, sideY), Image.LANCZOS)
        if args.overlay_alpha:
            ov.putalpha(args.overlay_alpha)
        st.overlay_rgba = ov
    st.side = (sideX, sideY)
    st.drawer = drawer
    st.perceptors = [P.Perceptor(st.session, i) for i in range(len(args.clip_models))]
    st.make_cutouts = P.MakeCutouts(clip_cfgs[0]["image_res"], args.num_cuts, st.session, cut_pow=args.cut_pow, seed=st.seed,
                                    aspect=aspect)

    # ---- prompts, in the order ascend_txt scores them (pixray.py:859-958): text, vector, noise; then image prompts
    tables = [[] for _ in args.clip_models]
    clip_embeds, clip_weights = [], []
    for prompt in args.prompts:
        for i, m in enumerate(args.clip_models):
            txt, weight, stop = P.parse_prompt(prompt)
            embed = _text_embed(args, m, txt, clip_cfgs[i]["out_dim"])
            if kind == E.DRAWER_VDIFF and m == drawer.clip_model:
                clip_embeds.append(embed)
                clip_weights.append(weight)
            tables[i].append(P.Prompt(embed, weight, stop))
    if kind == E.DRAWER_VDIFF and clip_embeds:  # pixray.py:880-885
        w = torch.tensor(clip_weights, dtype=torch.float32)
        drawer.set_clip_embed(torch.nn.functional.normalize(torch.cat(clip_embeds).mul(w[:, None]).sum(0, keepdim=True), dim=-1))
    for vect_prompt in args.vector_prompts:
        f1, weight, stop = P.parse_prompt(vect_prompt)
        weight = 0.1 * weight  # "vect_promts are by nature tuned to 10% of a normal prompt"
        table = _vector_table(f1)
        for i, m in enumerate(args.clip_models):
            if m not in table:
                print(f"WARNING: no vector for {m} in {f1}!")
                continue
            tables[i].append(P.Prompt(torch.tensor(np.array(table[m]), dtype=torch.float32), weight, stop))
    for seed, weight in zip(args.noise_prompt_seeds, args.noise_prompt_weights):
        gen = torch.Generator().manual_seed(seed)
        last = len(args.clip_models) - 1  # the reference appends to the loop's last perceptor (pixray.py:955-958)
        tables[last].append(P.Prompt(torch.empty([1, clip_cfgs[last]["out_dim"]]).normal_(generator=gen), weight))
    for i, t in enumerate(tables):
        if not t:
            raise ValueError(f"no prompts for perceptor {args.clip_models[i]}")
        P.Prompt.register(st.session, i, t)
    st.prompt_tables = tables
    # spot prompts (pixray.py:917-931): text Prompts scored on the cutouts of the masked image (fetch_spot_indexes, 370-394)
    spot_on, spot_off = split_pipes(args.spot_prompts) or [], split_pipes(args.spot_prompts_off) or []
    if spot_on or spot_off:
        eng.set_spot_mask(_spot_mask(args, clip_cfgs[0]["image_res"], aspect))
        for i, m in enumerate(args.clip_models):
            for which, plist in ((1, spot_on), (0, spot_off)):
                parsed = [P.parse_prompt(p) for p in plist]
                embeds = [_text_embed(args, m, txt, clip_cfgs[i]["out_dim"]) for (txt, _, _) in parsed]
                eng.set_spot_prompts(i, which, torch.cat(embeds).numpy() if embeds else [], [w for (_, w, _) in parsed],
                                     [s_ for (_, _, s_) in parsed])
    if args.image_prompts:
        imgs = [_load_image(p, sideX, sideY) for p in args.image_prompts]
        w = None if args.image_prompt_weight is None else [args.image_prompt_weight] * len(imgs)
        eng.set_image_prompts(imgs, w)  # each at its own (aspect-preserving) size

    # ---- anchors to the start (pixray.py:833-850, 1344-1375): image_labels, then the init_weight family, in ascend_txt's order
    _attach_anchors(args, st, drawer, sideX, sideY)

    # ---- filters: "name:weight,..." (pixray.py:651-668); they run inside the fused iteration, between synth and the cutouts
    st.filters = []
    if args.filters is not None:
        if kind == E.DRAWER_VDIFF:
            raise NotImplementedError("filters on the vdiff drawer are not built")
        for chunk in [c.strip() for c in args.filters.split(",")]:
            filt_name, weight, _ = P.parse_prompt(chunk)
            if filt_name not in filters_class_table:
                raise ValueError(f"Requested filter not found, aborting: {filt_name}")
            inst = filters_class_table[filt_name](args, device=eng.device)
            inst.attach(st.session, args, weight)
            st.filters.append({"filter": inst, "weight": weight})

    # ---- custom losses: "name:weight,name2->arg" (pixray.py:961-990)
    st.custom = []
    if args.custom_loss is not None:
        for chunk in [c.strip() for c in args.custom_loss.split(",")]:
            parts = chunk.split("->")
            loss_name, weight, _ = P.parse_prompt(parts[0])
            inst = loss_class_table[loss_name](device=eng.device)
            inst.instance_settings(parts[1:])
            st.custom.append({"loss": inst, "weight": weight})
        for t in st.custom:
            args = t["loss"].parse_settings(args)
        for t in st.custom:
            t["loss"].attach(st.session, args, t["weight"])
    st.cur_iteration, st.best_loss, st.best_iter, st.num_loss_drop = 0, 1e20, 0, 0
    st.max_loss_drops, st.iter_drop_delay = len(args.learning_rate_drops), 12
    st.loss_buf = np.zeros(eng.num_losses(), dtype=np.float32)
    st.losses = None
    if args.batches != 1:
        eng.set_batches(args.batches)  # pixray.py:1464-1482: gradient accumulation over several cutout draws
    rebuild_optimisers(args)
    # train()'s control decisions move to the device when the engine can take them (everything but vdiff, whose loop
    # rebuilds Adam with a scheduled rate every iteration on the host, pixray.py:1489-1495)
    st.managed = bool(getattr(args, "b200_device_checkdrop", True)) and hasattr(eng, "set_schedule") and kind != E.DRAWER_VDIFF
    if st.managed:
        eng.set_schedule(st.lr, st.iter_drop_delay, st.max_loss_drops, bool(args.auto_stop), list(args.learning_rate_drops)[:16])
        st.stop_iter = None
    return args


def _attach_anchors(args, st, drawer, sideX, sideY):
    eng = st.engine
    wants_z = args.init_weight or args.init_weight_dist or args.init_weight_cos
    if (wants_z or args.image_labels is not None) and not hasattr(eng, "add_anchor"):
        raise NotImplementedError("this engine build has no anchor losses (pxr_add_anchor)")
    if args.image_labels is not None:
        # one label latent: every file encoded (drawer.get_z_from_tensor), rows normalised along the last axis, averaged,
        # normalised as a whole (pixray.py:833-850)
        import glob
        from PIL import Image
        files = sorted(glob.glob(args.image_labels))
        if not files:
            raise FileNotFoundError(f"image_labels matched no file: {args.image_labels}")
        cur = []
        for f in files:
            rgb = Image.open(f).convert("RGB").resize((sideX, sideY), Image.LANCZOS)
            t = torch.from_numpy(np.asarray(rgb, dtype=np.float32) / 255.0).permute(2, 0, 1).unsqueeze(0) * 2 - 1
            cur.append(torch.as_tensor(drawer.get_z_from_tensor(t)).float().cpu())
        emb = torch.stack(cur)
        emb = emb / emb.norm(dim=-1, keepdim=True)
        emb = emb.mean(dim=0)
        emb = emb / emb.norm()
        eng.add_anchor(E.ANCHOR_SPHERICAL, args.image_label_weight, emb)
    if wants_z and st.z_orig is None:
        raise ValueError("init_weight needs an init_image (z_orig is the encoded init image, pixray.py:719)")
    if args.init_weight:
        eng.add_anchor(E.ANCHOR_SPHERICAL, args.init_weight, st.z_orig)
    if args.init_weight_dist:
        eng.add_anchor(E.ANCHOR_MSE, args.init_weight_dist, st.z_orig)
    if args.init_weight_pix:
        if st.init_image_tensor is None:
            print("OOPS IIT is 0")  # the reference's own message (pixray.py:1364-1365); the term is skipped there too
        else:
            eng.add_anchor(E.ANCHOR_PIX, args.init_weight_pix, st.init_image_tensor)
    if args.init_weight_cos:
        eng.add_anchor(E.ANCHOR_COS, args.init_weight_cos, st.z_orig)


def _spot_mask(args, cut_size, aspect):
    """fetch_spot_indexes (pixray.py:370-394): args.spot_file, else the reference's inputs/spot_wide.png (non-square canvas) /
    inputs/spot_square.png, as RGB, LANCZOS-resized to cut_size x cut_size, >= 0.5.  Arrays / tensors ([cs, cs] or
    [3, cs, cs], truthy inside the spot) are taken as they are."""
    src = getattr(args, "spot_file", None)
    if src is not None and not isinstance(src, (str, os.PathLike)):
        return np.asarray(src.cpu() if torch.is_tensor(src) else src) != 0
    if src is None:
        name = "spot_wide.png" if aspect != 1.0 else "spot_square.png"
        cands = [os.path.join("inputs", name)]
        if os.environ.get("PIXRAY_ROOT"):
            cands.append(os.path.join(os.environ["PIXRAY_ROOT"], "inputs", name))
        src = next((c for c in cands if os.path.exists(c)), None)
        if src is None:
            raise FileNotFoundError(f"spot prompts need a mask image: pass spot_file, or set PIXRAY_ROOT (tried {cands})")
    from PIL import Image
    img = Image.open(src).convert("RGB").resize((cut_size, cut_size), Image.LANCZOS)
    t = np.asarray(img, dtype=np.float32) / 255.0  # TF.to_tensor
    return np.ascontiguousarray(np.transpose(t, (2, 0, 1)) >= 0.5)


def _load_image(src, sideX, sideY):
    """Image.open(path).convert('RGB') -> resize_image(img, (sideX, sideY)) -> to_tensor (pixray.py:949-953, 514-518): the
    source aspect ratio is kept and the image is never upsampled beyond the canvas AREA; MakeCutouts pools whatever size
    comes out.  Tensors ([1|-, 3, h, w] in [0, 1]) are taken as they are."""
    if torch.is_tensor(src):
        return src.to(torch.float32).reshape(1, 3, *src.shape[-2:]).contiguous()
    from PIL import Image  # only needed for file image prompts
    img = Image.open(src).convert("RGB")
    ratio = img.size[0] / img.size[1]
    area = min(img.size[0] * img.size[1], sideX * sideY)
    size = round((area * ratio) ** 0.5), round((area / ratio) ** 0.5)
    img = img.resize(size, Image.LANCZOS)
    return torch.from_numpy(np.asarray(img, dtype=np.float32) / 255.0).permute(2, 0, 1).unsqueeze(0).contiguous()


def re_average_z(args):
    """pixray.py:1408-1420: render, paste the overlay, re-encode (drawer.reapply_from_tensor)."""
    from PIL import Image
    st = _state
    cur = st.drawer.to_image().convert("RGB")
    if st.overlay_rgba is not None:
        cur.paste(st.overlay_rgba, (0, 0), mask=st.overlay_rgba)
    cur = cur.resize(st.side, Image.LANCZOS)
    t = torch.from_numpy(np.asarray(cur, dtype=np.float32) / 255.0).permute(2, 0, 1).unsqueeze(0)
    st.drawer.reapply_from_tensor(t * 2 - 1)


def rebuild_optimisers(args):
    """pixray.py:520-555: a FRESH args.optimiser at learning_rate / 10^drops, or the drawer's own Adam and rate
    (fftdrawer.py:63-67)."""
    st = _state
    drop_divisor = 10 ** st.num_loss_drop
    own = st.drawer.get_opts(drop_divisor)
    st.lr = own[0]["lr"] if own else args.learning_rate / drop_divisor
    P.install_optimiser(st.engine, "Adam" if own else args.optimiser)
    return st.lr


def checkdrop(args, it, losses):
    """pixray.py:1090-1109."""
    st = _state
    loss_sum = float(sum(losses))
    if loss_sum < st.best_loss:
        st.best_loss, st.best_iter = loss_sum, it
        return False
    return (it - st.best_iter) >= st.iter_drop_delay


def train(args, cur_it):
    """pixray.py:1436-1512.  The whole iteration (synth -> cutouts -> encode -> losses -> backward -> optimiser step ->
    clip_z) is ONE pxr_iterate call.  Default: checkdrop, the scheduled learning-rate drops and auto-stop are decided inside that
    call on the device (pxr_set_schedule) and the host only POLLS a pinned status record -- no synchronisation in the
    loop; iterations enqueued after the device raised `stopped` leave z untouched, so the result equals the reference's
    control flow.  With b200_device_checkdrop=False (and for vdiff) the reference's host-side flow runs as written, one
    loss readback per iteration."""
    st = _state
    if getattr(st, "managed", False):
        return _train_managed(args, cur_it)
    rebuild = False
    if cur_it < args.iterations:
        if apply_overlay(args, cur_it):
            re_average_z(args)
        st.session.begin_iteration(cur_it)
        drawer, eng = st.drawer, st.engine
        if isinstance(drawer, P.VdiffDrawer):
            eng.vdiff_set_iteration(cur_it)
        eng.iterate(drawer.get_z(), st.lr, cur_it, params=None, losses_out=st.loss_buf)
        st.losses = st.loss_buf.copy()
        if cur_it in args.learning_rate_drops:
            print("Dropping learning rate")
            rebuild = True
        else:
            did_drop = checkdrop(args, cur_it, st.losses)
            if args.auto_stop is True:
                rebuild = did_drop
    if isinstance(st.drawer, P.VdiffDrawer) and cur_it >= 1:  # pixray.py:1489-1495: a fresh Adam whatever args.optimiser
        lr = float(st.drawer.sigmas[cur_it] / st.drawer.alphas[cur_it])
        st.drawer.makenoise(cur_it)
        st.lr = min(lr * 0.001, 0.01)
        P.install_optimiser(st.engine, "Adam")
    if cur_it == args.iterations:
        checkin(args, cur_it, st.losses)
        return False
    if rebuild:
        st.num_loss_drop += 1
        if st.num_loss_drop > st.max_loss_drops:
            return False
        st.best_iter, st.best_loss = cur_it, 1e20
        rebuild_optimisers(args)
    return True


def _absorb_status(rec):
    st = _state
    st.losses = rec["losses"]
    st.best_loss, st.best_iter, st.num_loss_drop, st.lr = rec["best_loss"], rec["best_iter"], rec["num_loss_drop"], rec["lr"]
    if rec["stopped"] and st.stop_iter is None:
        st.stop_iter = rec["iter"]


def _train_managed(args, cur_it):
    st = _state
    if cur_it < args.iterations:
        if apply_overlay(args, cur_it):
            re_average_z(args)
        st.session.begin_iteration(cur_it)
        if cur_it in args.learning_rate_drops:
            print("Dropping learning rate")
        st.engine.iterate(st.drawer.get_z(), st.lr, cur_it, params=None, losses_out=None)
        rec = st.engine.poll_status()  # the last COMPLETED iteration (lags the launch by the queue depth): no sync
        if rec is not None:
            _absorb_status(rec)
            if st.stop_iter is not None:
                # train() returned False at stop_iter; what was enqueued since did not move z.  Rewind the counter to
                # that call (do_run then counts it like the reference does).
                st.engine.sync()
                st.cur_iteration = st.stop_iter
                return False
    if cur_it == args.iterations:
        st.engine.sync()
        rec = st.engine.poll_status()
        if rec is not None:
            _absorb_status(rec)
        checkin(args, cur_it, st.losses)
        return False
    return True


def checkin(args, it, losses):
    """The final save of pixray.py:1158-1201 (intermediate frames, PNG metadata and video are I/O outside the scope)."""
    st = _state
    st.image = st.drawer.synth(it).detach().clamp(0, 1).cpu()
    outdir = getattr(args, "outdir", None)
    if outdir and "%" not in outdir:
        try:
            from PIL import Image
            os.makedirs(outdir, exist_ok=True)
            arr = (st.image[0].permute(1, 2, 0).numpy() * 255).astype(np.uint8)
            Image.fromarray(arr, mode="RGB").save(os.path.join(outdir, args.output))
        except ImportError:
            pass


def do_run(args, return_display=False):
    """pixray.py:1517-1638, the non-animation branch: loop train() until it says stop; RuntimeError gets the reference's
    memory hint and is re-raised, KeyboardInterrupt ends the loop cleanly."""
    st = _state
    try:
        keep_going = True
        while keep_going:
            try:
                keep_going = train(args, st.cur_iteration)
                if st.cur_iteration == args.iterations:
                    break
                st.cur_iteration += 1
                if keep_going and return_display and st.cur_iteration % args.display_every == 0:
                    return False
            except RuntimeError as e:
                print("Oops: runtime error: ", e)
                print("Try reducing --num-cuts to save memory")
                raise e
    except KeyboardInterrupt:
        pass
    return True


def save_checkpoint(path):
    """z, Adam state, learning-rate / drop bookkeeping and the iteration counter of the running session, for resume."""
    st = _state
    st.engine.sync()
    with open(path, "wb") as f:
        blob = st.engine.save_state()
        f.write(int(st.cur_iteration).to_bytes(8, "little"))
        f.write(int(st.num_loss_drop).to_bytes(8, "little"))
        f.write(np.float64(st.lr).tobytes())
        f.write(blob)


def load_checkpoint(path):
    """Into a session built by do_init with the same settings: restores z / Adam / bookkeeping; do_run then continues from the
    saved iteration."""
    st = _state
    with open(path, "rb") as f:
        raw = f.read()
    st.cur_iteration = int.from_bytes(raw[:8], "little")
    st.num_loss_drop = int.from_bytes(raw[8:16], "little")
    st.lr = float(np.frombuffer(raw[16:24], dtype=np.float64)[0])
    st.engine.load_state(raw[24:])
    st.drawer.set_z(st.engine.read_z())
    return st.cur_iteration


def get_image():
    """[1, 3, H, W] in [0, 1]: the image of the last checkin."""
    return getattr(_state, "image", None)


def run(prompts=None, drawer="vqgan", **kwargs):
    """One-stop call from notebooks or other python code (pixray.py:2115-2120)."""
    reset_settings()
    add_settings(prompts=prompts, drawer=drawer, **kwargs)
    settings = apply_settings()
    do_init(settings)
    do_run(settings)
