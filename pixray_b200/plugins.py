"""pixray's plugin surface (SURVEY.md 8b) on top of the B200 engine.

Same class / method names, argument meaning and error behaviour as the reference, so a pixray loop written against
`drawer.synth`, `MakeCutouts.__call__`, `perceptor.encode_image`, `Prompt.__call__`, `opt.step()` / `drawer.clip_z()`
runs unchanged -- each method forwards to one C entry point (include/pixray_b200.h).  Like the reference's module
globals (pixray.py:1022-1063) there is ONE session per process: the plugin objects share one `B200Engine`.

Gradients do not flow through torch autograd here: the engine owns the hand-written backward chain, so
`Session.backward()` replaces `sum(lossAll).backward()` (pixray.py:1481-1482) and writes `drawer.z.grad`.
"""
import math

import numpy as np
import torch
from torch.nn import functional as F

from . import cutouts as cut_sampler
from . import engine as E


class DrawingInterface:
    """DrawingInterface.py:1-12 -- the declared part of the drawer contract."""

    @staticmethod
    def add_settings(parser):
        return parser

    def __init__(self, settings):
        self.settings = settings

    def load_model(self, settings, device):
        pass

    @torch.no_grad()
    def to_image(self):
        """TF.to_pil_image(self.synth(None)[0].cpu()) (vqgan.py:197-200 and the other drawers): float -> mul(255).byte()."""
        from PIL import Image
        out = self.synth(None)
        return Image.fromarray(out[0].detach().cpu().mul(255).byte().permute(1, 2, 0).numpy(), mode="RGB")


class Session:
    """The shared engine + the per-iteration state the reference keeps in globals (cur_iteration,
    global_padding_mode, global_fill_color: pixray.py:1250-1258)."""

    def __init__(self, eng: E.B200Engine):
        self.engine = eng
        self.cur_iteration = 0
        self.global_padding_mode = "reflection"
        self.global_fill_color = 0.0
        self.last_embeds = {}  # clip_idx -> the tensor Perceptor.encode_image handed out this iteration

    def begin_iteration(self, cur_iteration, fill=None, rng=None):
        self.cur_iteration = cur_iteration
        self.global_padding_mode = "reflection" if cur_iteration % 2 == 0 else "border"  # pixray.py:1250-1253
        self.global_fill_color = float((rng or np.random).random()) if fill is None else float(fill)  # 1255-1258

    def backward(self, drawer):
        """loss.backward(): z.grad += d(sum of prompt losses)/dz (pixray.py:1481-1482)."""
        g = self.engine.backward()
        z = drawer.get_z()
        z.grad = g if z.grad is None else z.grad + g
        return g


class VqganDrawer(DrawingInterface):
    """vqgan.py:81-218 (synth 190-195, clip_z 202-204, get_z/set_z/get_z_copy 206-216)."""

    @staticmethod
    def add_settings(parser):
        parser.add_argument("--vqgan_model", type=str, help="VQGAN model", default="imagenet_f16_16384", dest="vqgan_model")
        return parser

    def __init__(self, settings, session: Session):
        super().__init__(settings)
        self.session = session
        self.z = None

    def load_model(self, settings, device):
        self.device = device
        lo, hi = self.session.engine.z_bounds()
        self.z_min, self.z_max = lo[None, :, None, None], hi[None, :, None, None]  # vqgan.py:141-142

    def get_opts(self, decay_divisor):
        return None  # engine builds Adam on get_z(), like pixray.py:537-539

    def get_num_resolutions(self):
        return self.session.engine.cfg.n_levels

    def init_from_tensor(self, init_tensor):
        """self.z, *_ = self.model.encode(init_tensor) (vqgan.py:174-176): taming Encoder + quant_conv + nearest code on the
        engine (pxr_vqgan_encode)."""
        self.z = self.get_z_from_tensor(init_tensor).clone()
        return self.z

    def reapply_from_tensor(self, new_tensor):
        new_z = self.get_z_from_tensor(new_tensor)
        with torch.no_grad():
            self.z.copy_(new_z)

    def get_z_from_tensor(self, ref_tensor):
        return self.session.engine.vqgan_encode(ref_tensor)

    def synth(self, cur_iteration):
        return self.session.engine.synth(self.z)

    def clip_z(self):
        with torch.no_grad():
            self.z.copy_(self.z.maximum(self.z_min).minimum(self.z_max))

    def get_z(self):
        return self.z

    def set_z(self, new_z):
        if self.z is None:
            self.z = new_z.detach().to(self.session.engine.device, torch.float32).contiguous().clone()
            return self.z
        with torch.no_grad():
            return self.z.copy_(new_z)

    def get_z_copy(self):
        return self.z.clone()


class FastPixelDrawer(DrawingInterface):
    """fast_pixeldrawer.py:24-110: z = colour grid, synth = nearest upsample + clamp_with_grad."""

    @staticmethod
    def add_settings(parser):
        parser.add_argument("--pixel_size", nargs=2, type=int, help="Pixel size (width height)", default=None, dest="pixel_size")
        parser.add_argument("--pixel_scale", type=float, help="Pixel scale", default=None, dest="pixel_scale")
        return parser

    @staticmethod
    def grid_for(size, pixel_size=None, pixel_scale=None, verbose=True):
        """(num_rows, num_cols) as FastPixelDrawer.__init__ derives them (fast_pixeldrawer.py:37-63): an explicit
        pixel_size (width, height), else 40x40 on a square canvas, 40x50 on a portrait one, 80x45 on a landscape one; divided
        by pixel_scale; never larger than the canvas."""
        canvas_width, canvas_height = size
        if pixel_size is not None:
            num_cols, num_rows = pixel_size
        elif canvas_width == canvas_height:
            num_cols, num_rows = 40, 40
        elif canvas_width < canvas_height:
            num_cols, num_rows = 40, 50
        else:
            num_cols, num_rows = 80, 45
        if pixel_scale is not None and pixel_scale > 0:
            num_cols, num_rows = int(num_cols / pixel_scale), int(num_rows / pixel_scale)
        shrink = False
        if num_cols > canvas_width:
            shrink, num_cols = True, canvas_width
        if num_rows > canvas_height:
            shrink, num_rows = True, canvas_height
        if shrink and verbose:
            print("pixel grid size should not be larger than output pixel size: reducing pixel grid")
        return num_rows, num_cols

    def __init__(self, settings, session: Session):
        super().__init__(settings)
        self.session = session
        self.pixel_size = (session.engine.z_shape[2], session.engine.z_shape[3])
        self.output_size = session.engine.image_hw
        self.num_rows, self.num_cols = self.pixel_size
        self.z = None

    def get_opts(self, decay_divisor):
        return None

    def get_num_resolutions(self):
        return None

    def get_z_from_tensor(self, ref_tensor):
        return F.interpolate((ref_tensor + 1) / 2, size=self.pixel_size, mode="bilinear", align_corners=False)

    def init_from_tensor(self, init_tensor):
        self.z = self.get_z_from_tensor(init_tensor).to(self.session.engine.device, torch.float32).contiguous()

    def synth(self, cur_iteration):
        return self.session.engine.synth(self.z)

    def clip_z(self):
        with torch.no_grad():
            self.z.copy_(self.z.clip(0, 1))

    def get_z(self):
        return self.z

    def set_z(self, new_z):
        with torch.no_grad():
            return self.z.copy_(new_z)

    def get_z_copy(self):
        return self.z.clone()


class VdiffDrawer(DrawingInterface):
    """vdiff.py:58-190 (cc12m_1): z = the noisy image x; synth = one v-prediction step + ClampWithGrad; after every
    optimiser step the loop re-noises x (`makenoise`, pixray.py:1489-1495) and builds a fresh Adam."""

    @staticmethod
    def add_settings(parser):
        parser.add_argument("--vdiff_model", type=str, help="VDIFF model from [yfcc_2, yfcc_1, cc12m_1, cc12m_1_cfg]", default="yfcc_2", dest="vdiff_model")
        parser.add_argument("--vdiff_schedule", type=str, help="VDIFF schedule [default, log]", default="default", dest="vdiff_schedule")
        parser.add_argument("--vdiff_skip", type=float, help="skip a percentage of the way into the decay schedule (0-100)", default=0, dest="vdiff_skip")
        return parser

    def __init__(self, settings, session: Session):
        super().__init__(settings)
        self.session = session
        self.iterations = settings.iterations
        self.vdiff_skip = getattr(settings, "vdiff_skip", 0)
        if getattr(settings, "vdiff_schedule", "default") != "default":
            raise NotImplementedError("only the default (spliced DDPM/cosine) schedule is implemented")
        self.clip_model = "ViT-B/16"  # cc12m_1.py:111
        self.x = None

    def load_model(self, settings, device):
        self.device = device

    def get_opts(self, decay_divisor):
        return None

    def get_num_resolutions(self):
        return None

    def init_from_tensor(self, init_tensor, seed=None):
        from .util import vdiff_schedule
        eng = self.session.engine
        self.steps, self.alphas, self.sigmas = vdiff_schedule(self.iterations, self.vdiff_skip)
        eng.vdiff_set_schedule(self.steps, self.alphas, self.sigmas)
        g = None if seed is None else torch.Generator(device=eng.device).manual_seed(seed)
        self.x = torch.randn(eng.z_shape, device=eng.device, generator=g)
        if init_tensor is not None:  # vdiff.py:143: x = init * alpha_0 + noise * sigma_0
            self.x = init_tensor.to(eng.device) * float(self.alphas[0]) + self.x * float(self.sigmas[0])
        self.x = self.x.contiguous()

    def set_clip_embed(self, clip_embed):
        """sample_state[3] = {"clip_embed": ...} (pixray.py:880-885)."""
        self.session.engine.vdiff_set_clip_embed(torch.as_tensor(clip_embed).detach().cpu().numpy())

    def makenoise(self, cur_it):
        noise = torch.randn_like(self.x)
        return self.session.engine.vdiff_renoise(self.x, cur_it, noise)

    def synth(self, cur_iteration):
        self.session.engine.vdiff_set_iteration(cur_iteration)
        return self.session.engine.synth(self.x)

    def clip_z(self):
        return None

    def get_z(self):
        return self.x

    def set_z(self, new_z):
        with torch.no_grad():
            return self.x.copy_(new_z)

    def get_z_copy(self):
        return self.x.clone()


class FftDrawer(DrawingInterface):
    """fftdrawer.py:13-109, `fft_use="fft"`: params = the rfft2 spectrum [1, 3, H, W/2+1, 2] ~ N(0, 0.01^2)
    (aphantasia fft_image), synth = to_valid_rgb(fft_image)(contrast=0.9); the drawer owns its Adam (lr fft_lrate /
    decay_divisor, fftdrawer.py:63-67), which `get_opts` reports as a learning rate for the engine's fused Adam."""

    @staticmethod
    def add_settings(parser):
        parser.add_argument("--fft_use", type=str, help="use fft or dwt or pixel", default="fft", dest="fft_use")
        parser.add_argument("--fft_decay", default=1.5, type=float, dest="fft_decay")
        parser.add_argument("--fft_wave", default="coif2", help="wavelets: db[1..], coif[1..], haar, dmey", dest="fft_wave")
        parser.add_argument("--fft_sharp", default=0.3, type=float, dest="fft_sharp")
        parser.add_argument("--fft_colors", default=1.5, type=float, dest="fft_colors")
        parser.add_argument("--fft_lrate", default=0.3, type=float, help="Learning rate", dest="fft_lrate")
        return parser

    def __init__(self, settings, session: Session):
        super().__init__(settings)
        self.session = session
        if getattr(settings, "fft_use", "fft") != "fft":
            raise NotImplementedError("fft_use: only 'fft' is on the hot-path scope (dwt / pixel need pytorch_wavelets)")
        self.lrate = getattr(settings, "fft_lrate", 0.3)
        self.params = None

    def load_model(self, settings, device):
        self.device = device

    def get_opts(self, decay_divisor=1):
        return [{"lr": self.lrate / decay_divisor}]

    def get_num_resolutions(self):
        return None

    def init_from_tensor(self, init_tensor, seed=None):
        if init_tensor is not None:
            raise NotImplementedError("resuming the spectrum from an image (fft_image(resume=...)) is init-time and not built")
        eng = self.session.engine
        g = None if seed is None else torch.Generator(device=eng.device).manual_seed(seed)
        self.params = (0.01 * torch.randn(eng.z_shape, device=eng.device, generator=g)).contiguous()  # fft_image(sd=0.01)

    def synth(self, cur_iteration):
        return self.session.engine.synth(self.params)

    def clip_z(self):
        pass

    def get_z(self):
        return self.params  # the reference returns None here and optimises self.params through its own Adam

    def set_z(self, new_z):
        with torch.no_grad():
            return self.params.copy_(new_z)

    def get_z_copy(self):
        return self.params.clone()


class MakeCutouts:
    """pixray.py:399-511.  `transforms` is the per-iteration cache of composed 3x3s (pixray.py:498); when it is None
    a fresh set is sampled (the distributions of the reference's augmentation stacks, pixray_b200/cutouts.py)."""

    def __init__(self, cut_size, cutn, session: Session, cut_pow=1.0, seed=0, aspect=1.0):
        self.cut_size, self.cutn, self.cut_pow = cut_size, cutn, cut_pow
        self.aspect = aspect  # global_aspect_width (pixray.py:402, 1931)
        self.cutn_zoom = int(0.6 * cutn)
        self.noise_fac = 0.1
        self.transforms = None
        self.color_jitter = None
        self.session = session
        self._rng = np.random.default_rng(seed)

    def __call__(self, input, spot=None):
        return self.forward(input, spot)

    def forward(self, input, spot=None):
        if spot is not None:
            raise NotImplementedError("spot prompts are off by default and out of scope (SURVEY.md 8f-2)")
        s = self.session
        if self.transforms is None:
            self.transforms = torch.from_numpy(
                cut_sampler.sample_transforms(self.cutn, self.cut_size, int(self._rng.integers(1 << 31)), aspect=self.aspect))
            # the live stacks end in K.ColorJitter (pixray.py:416, 436); replays of the cached transforms within the
            # same iteration (pixray.py:480-486) do not repeat it
            jitter = cut_sampler.sample_color_jitter(self.cutn, int(self._rng.integers(1 << 31)))
        else:
            jitter = None
        self.color_jitter = jitter
        pad = E.PAD_REFLECTION if s.global_padding_mode == "reflection" else E.PAD_BORDER
        facs = noise = None
        if self.noise_fac:
            facs = (self._rng.random(self.cutn) * self.noise_fac).astype(np.float32)        # pixray.py:509
            noise = torch.randn(self.cutn, 3, self.cut_size, self.cut_size, device=s.engine.device)  # pixray.py:510
        return s.engine.make_cutouts(input, transforms=self.transforms.numpy(), zoom_padding=pad,
                                     fill=s.global_fill_color, noise_facs=facs, noise=noise, it=s.cur_iteration,
                                     color_jitter=jitter)


class Perceptor:
    """CLIP_Base surface (slip.py:44-74): input_resolution, output_dim, encode_image -> unit-norm [N, D]."""

    def __init__(self, session: Session, clip_idx=0):
        self.session, self.clip_idx = session, clip_idx
        self.device = session.engine.device
        c = session.engine.cfg.clip[clip_idx]
        self.input_resolution, self.output_dim = c.image_res, c.out_dim

    def encode_image(self, imgs, input_range=None, apply_preprocess=True):
        if input_range is not None or not apply_preprocess:
            raise NotImplementedError("only the default preprocess path of the hot loop is implemented (pixray.py:1295)")
        e = self.session.engine.encode_image(self.clip_idx, imgs)
        self.session.last_embeds[self.clip_idx] = e
        return e

    def encode_text(self, text):
        raise NotImplementedError("text towers are init-time (SURVEY.md row 10); pass prompt embeddings")


class Prompt:
    """pixray.py:268-280.  Instances register themselves with the engine so the loss and its gradient stay on device."""

    def __init__(self, embed, weight=1.0, stop=float("-inf")):
        self.embed = torch.as_tensor(embed, dtype=torch.float32).reshape(-1, torch.as_tensor(embed).shape[-1])
        self.weight = torch.as_tensor(float(weight))
        self.stop = torch.as_tensor(float(stop))
        self._session, self._clip_idx, self._index = None, 0, 0

    @staticmethod
    def register(session: Session, clip_idx, prompts):
        """pmsTable[clip_model] = [Prompt, ...] (pixray.py:859-915)."""
        if any(p.embed.shape[0] != 1 for p in prompts):
            raise ValueError("one embedding row per registered Prompt; image prompts ([cutn, D] rows, refreshed every "
                             "iteration) go through engine.set_image_prompts")
        session.engine.set_prompts(clip_idx, torch.cat([p.embed for p in prompts]).numpy(),
                                   [float(p.weight) for p in prompts], [float(p.stop) for p in prompts])
        for i, p in enumerate(prompts):
            p._session, p._clip_idx, p._index = session, clip_idx, i

    def __call__(self, input):
        return self.forward(input)

    def forward(self, input):
        if self._session is None:
            raise RuntimeError("Prompt.register(session, clip_idx, prompts) must be called first")
        # `input` is normally the tensor perceptor.encode_image just returned (possibly through .float()): the engine still
        # holds those embeddings un-normalised, which its backward needs, so they are not passed back in.  Foreign
        # embeddings are scored as given into scratch buffers: they have no graph behind them, and the engine's own
        # embeddings / gradient (what Session.backward() propagates) are left untouched.
        own = self._session.last_embeds.get(self._clip_idx)
        mine = own is not None and input.data_ptr() == own.data_ptr() and input.shape == own.shape
        return self._session.engine.prompt_loss(self._clip_idx, None if mine else input)[self._index]


def parse_prompt(prompt):
    """pixray.py:290-321: text, text:weight or text:weight:stop."""
    def is_number(s):
        try:
            float(s)
            return True
        except ValueError:
            return False

    text, weight, stop = prompt, 1, float("-inf")
    extra = []
    keep = True
    while len(extra) < 2 and keep:
        vals = text.rsplit(":", 1)
        if len(vals) > 1 and is_number(vals[1]):
            extra.append(float(vals[1]))
            text = vals[0]
        else:
            keep = False
    if len(extra) == 1:
        weight = extra[0]
    elif len(extra) == 2:
        weight, stop = extra[1], extra[0]
    return text, weight, stop


from .util import get_learning_rate_drops  # noqa: E402,F401  (pixray.py:1999-2003)


def install_optimiser(engine, name):
    """A fresh optimiser `name` (Adam, AdamW, Adagrad, Adamax or DiffGrad) on the engine.  The engine switches kind only
    when `name` differs from its current one; otherwise this is a plain reset of the current optimiser's state."""
    if name != getattr(engine, "optimizer", "Adam"):
        engine.set_optimizer(name)
    else:
        engine.reset_optimizer()


class Optimizer:
    """optim.<optimiser>([drawer.get_z()], lr) as rebuild_optimisers builds it (pixray.py:520-555): zero_grad / step.
    optimiser: Adam, AdamW, Adagrad, Adamax or DiffGrad, each with its library's defaults."""

    def __init__(self, session: Session, drawer, lr, optimiser="Adam"):
        self.session, self.drawer, self.lr = session, drawer, lr
        install_optimiser(session.engine, optimiser)

    def zero_grad(self):
        z = self.drawer.get_z()
        z.grad = None

    def step(self):
        z = self.drawer.get_z()
        if getattr(z, "grad", None) is not None:  # the gradient the loop accumulated (several passes when batches > 1)
            self.session.engine.set_z_grad(z.grad.contiguous())
        self.session.engine.step(z, self.lr, self.session.cur_iteration)


def train_iteration(session: Session, drawer, make_cutouts, perceptors, prompt_table, opt):
    """The body of train()/ascend_txt for the default settings (pixray.py:1243-1406, 1436-1512), expressed with the
    plugin objects exactly like the reference does.  Returns the list of scalar losses."""
    opt.zero_grad()
    out = drawer.synth(session.cur_iteration)
    cutouts = make_cutouts(out)
    result = []
    for i, perceptor in enumerate(perceptors):
        iii = perceptor.encode_image(cutouts).float()
        for prompt in prompt_table[i]:
            result.append(prompt(iii))
    make_cutouts.transforms = None  # clear the per-iteration cache (pixray.py:1339-1342)
    session.backward(drawer)
    opt.step()
    drawer.clip_z()
    if isinstance(drawer, VdiffDrawer) and session.cur_iteration >= 1:
        # pixray.py:1489-1495: re-noise x for the next timestep and start a fresh Adam (whatever the optimiser setting)
        # with the schedule's step size
        it = session.cur_iteration
        lr = float(drawer.sigmas[it] / drawer.alphas[it])
        drawer.makenoise(it)
        opt.lr = min(lr * 0.001, 0.01)
        install_optimiser(session.engine, "Adam")
    return result
