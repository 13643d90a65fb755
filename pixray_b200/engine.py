"""Python face of the C-ABI engine (include/pixray_b200.h).

torch is used only for device memory: tensors are handed to the library as raw device pointers.  Every method
maps 1:1 onto a C entry point, which in turn replaces one method of the reference's loop (see the header).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

DRAWER_VQGAN, DRAWER_PIXEL, DRAWER_FFT, DRAWER_VDIFF = 0, 1, 2, 3
LOSS_SYMMETRY, LOSS_SATURATION, LOSS_PALETTE, LOSS_SMOOTHNESS, LOSS_EDGE, LOSS_GAUSSIAN, LOSS_AESTHETIC = range(7)
ANCHOR_SPHERICAL, ANCHOR_MSE, ANCHOR_COS, ANCHOR_PIX = 0, 1, 2, 3
FILTER_TILER, FILTER_WALLPAPER, FILTER_LOOKUP = range(3)
PAD_REFLECTION, PAD_BORDER = 0, 1
MOD_VQGAN, MOD_CLIP0, MOD_CLIP1 = 0, 1, 2
# args.optimiser (pixray.py:536-553) -> PXR_OPT_*; each with its library's defaults, only lr is set
OPTIMISERS = {"Adam": 0, "AdamW": 1, "Adagrad": 2, "Adamax": 3, "DiffGrad": 4}

VQGAN_F16_16384 = dict(z_channels=256, n_embed=16384, ch=128, ch_mult=(1, 1, 2, 2, 4), num_res_blocks=2,
                       attn_resolution=16, resolution=256)
CLIP_ARCH = {
    "ViT-B/32": dict(width=768, layers=12, heads=12, patch=32, image_res=224, out_dim=512),
    "ViT-B/16": dict(width=768, layers=12, heads=12, patch=16, image_res=224, out_dim=512),
    "ViT-L/14": dict(width=1024, layers=24, heads=16, patch=14, image_res=224, out_dim=768),
}


class EngineError(RuntimeError):
    pass


class B200Engine:
    def __init__(self, *, drawer=DRAWER_VQGAN, image_hw=(256, 256), vqgan=None, grid=None, cutn=64, cut_size=224,
                 clip=(), noise_fac=0.1, seed=0, device=0, rank=0, world=1, grad_scale=0.0, lr_betas=(0.9, 0.999),
                 adam_eps=1e-8, fft_decay=0.0, fft_colors=0.0, fft_contrast=0.0, cut_aspect=1.0):
        if not torch.cuda.is_available():
            raise EngineError("pixray_b200 needs a CUDA device (B200); there is no CPU fallback")
        self.lib = _lib.load()
        cfg = _lib.Config()
        cfg.device, cfg.rank, cfg.world = device, rank, world
        cfg.drawer = drawer
        cfg.image_h, cfg.image_w = image_hw
        if drawer == DRAWER_VQGAN:
            v = dict(VQGAN_F16_16384) if vqgan is None else dict(vqgan)
            cfg.z_channels, cfg.n_embed, cfg.ch = v["z_channels"], v["n_embed"], v["ch"]
            cfg.num_res_blocks, cfg.attn_resolution, cfg.resolution = v["num_res_blocks"], v["attn_resolution"], v["resolution"]
            cfg.n_levels = len(v["ch_mult"])
            for i, m in enumerate(v["ch_mult"]):
                cfg.ch_mult[i] = m
            f = 2 ** (cfg.n_levels - 1)
            self.z_shape = (1, cfg.z_channels, image_hw[0] // f, image_hw[1] // f)
        elif drawer == DRAWER_VDIFF:
            # VdiffDrawer's x (vdiff.py:118): [1, 3, gen_height, gen_width]
            self.z_shape = (1, 3, image_hw[0], image_hw[1])
        elif drawer == DRAWER_FFT:
            # FftDrawer params (fftdrawer.py:57-61): rfft2 spectrum [1, 3, H, W/2+1, 2]
            self.z_shape = (1, 3, image_hw[0], image_hw[1] // 2 + 1, 2)
        else:
            cfg.grid_rows, cfg.grid_cols = grid
            self.z_shape = (1, 3, grid[0], grid[1])
        cfg.cutn, cfg.cut_size = cutn, cut_size
        cfg.n_clip = len(clip)
        for i, c in enumerate(clip):
            for k, val in c.items():
                setattr(cfg.clip[i], k, val)
        cfg.noise_fac, cfg.seed = noise_fac, seed
        cfg.op_dtype, cfg.grad_scale = 0, grad_scale
        cfg.beta1, cfg.beta2, cfg.adam_eps = lr_betas[0], lr_betas[1], adam_eps
        cfg.fft_decay, cfg.fft_colors, cfg.fft_contrast = fft_decay, fft_colors, fft_contrast  # 0 -> 1.5 / 1.5 / 0.9
        cfg.cut_aspect = float(cut_aspect)  # global_aspect_width (pixray.py:1931); 1 = square canvas
        self.cut_aspect = float(cut_aspect)
        if self.cut_aspect != 1.0:  # the stretched source size in Python double arithmetic, like the reference computes it
            from .cutouts import source_size
            cfg.cut_src_h, cfg.cut_src_w = source_size(cut_size, self.cut_aspect)
        self.cfg = cfg
        self.device = torch.device("cuda", device)
        self.cutn, self.cut_size, self.world, self.rank = cutn, cut_size, world, rank
        self.n_local = cutn // world
        self.image_hw = tuple(image_hw)
        self.clip_dims = [c["out_dim"] for c in clip]
        self.n_prompts = [0 for _ in clip]  # loss slots per perceptor: text prompts + image prompts
        self._n_text = [0 for _ in clip]
        self._n_spot = [[0, 0] for _ in clip]  # [spot off, spot] prompts per perceptor (scored in the fused path only)
        self._n_img = 0
        h = C.c_void_p()
        rc = self.lib.pxr_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise EngineError(f"pxr_create failed ({rc}): {self.lib.pxr_last_error(None).decode()}")
        self.h = h
        self._keep = []
        self._ext = None  # torch view of the engine's stream (ordering against torch-side producers of z / noise)
        self.optimizer = "Adam"  # the kind pxr_create starts with; set_optimizer changes it

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc, what):
        if rc != 0:
            raise EngineError(f"{what} failed ({rc}): {self.lib.pxr_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.pxr_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._check(self.lib.pxr_sync(self.h), "pxr_sync")

    @staticmethod
    def _p(t):
        return None if t is None else C.c_void_p(t.data_ptr())

    def _p_inplace(self, t, what):
        """Raw pointer of a tensor the library reads AND writes in place: it must be a dense, contiguous fp32 CUDA
        tensor (the C ABI sees plain NCHW memory; a permuted-stride tensor would be silently misread)."""
        if t is None:
            return None
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise EngineError(f"{what} must be a contiguous float32 CUDA tensor (got dtype={t.dtype}, "
                              f"device={t.device}, strides={tuple(t.stride())})")
        return C.c_void_p(t.data_ptr())

    def _new(self, *shape):
        return torch.empty(*shape, device=self.device, dtype=torch.float32)

    # ------------------------------------------------------------------ setup
    def load_module(self, module_id, state_dict):
        """Feed a reference-style state_dict (taming VQModel or openai-CLIP 'visual.*' keys)."""
        for name, t in state_dict.items():
            if not torch.is_floating_point(t):
                continue
            a = t.detach().to(torch.float32).contiguous().cpu()
            dims = (C.c_int64 * max(a.dim(), 1))(*(a.shape if a.dim() else (1,)))
            rc = self.lib.pxr_load_weight(self.h, module_id, name.encode(), C.c_void_p(a.data_ptr()), dims,
                                          max(a.dim(), 1))
            self._check(rc, f"pxr_load_weight({name})")

    def finalize(self):
        self._check(self.lib.pxr_finalize(self.h), "pxr_finalize")

    def set_prompts(self, clip_idx, embeds, weights, stops):
        e = np.ascontiguousarray(np.asarray(embeds, dtype=np.float32))
        w = np.ascontiguousarray(np.asarray(weights, dtype=np.float32))
        s = np.ascontiguousarray(np.asarray(stops, dtype=np.float32))
        s = np.maximum(s, np.float32(-3.0e38))  # -inf -> lowest finite (maximum(d, -inf) == d either way)
        n, D = e.shape
        rc = self.lib.pxr_set_prompts(self.h, clip_idx, e.ctypes.data_as(C.c_void_p), n, D,
                                      w.ctypes.data_as(C.c_void_p), s.ctypes.data_as(C.c_void_p))
        self._check(rc, "pxr_set_prompts")
        self._n_text[clip_idx] = n
        self.n_prompts[clip_idx] = n + self._n_img

    def set_image_prompts(self, imgs, weights=None):
        """Image prompts (pixray.py:1308-1336): target images in [0, 1], each [1|-, 3, h, w] at ITS OWN size (a list), or one
        [n, 3, H, W] tensor.  Every iteration each is cut with that iteration's cached transforms, encoded by every
        perceptor and scored as a throwaway Prompt(embed [cutn, D], weight) appended after the perceptor's text prompts.
        n = 0 clears them."""
        if imgs is None or len(imgs) == 0:
            items = []
        elif torch.is_tensor(imgs):
            items = [t for t in torch.as_tensor(imgs, dtype=torch.float32).reshape(-1, 3, *imgs.shape[-2:])]
        else:
            items = [torch.as_tensor(t, dtype=torch.float32).reshape(3, *t.shape[-2:]) for t in imgs]
        items = [t.contiguous().cpu() for t in items]
        n = len(items)
        ptrs = (C.c_void_p * max(n, 1))(*[t.data_ptr() for t in items])
        hs = (C.c_int * max(n, 1))(*[t.shape[1] for t in items])
        ws = (C.c_int * max(n, 1))(*[t.shape[2] for t in items])
        wp = None
        if n and weights is not None:
            w = np.ascontiguousarray(np.asarray(weights, dtype=np.float32).reshape(n))
            wp = w.ctypes.data_as(C.c_void_p)
        self._check(self.lib.pxr_set_image_prompts_sized(self.h, ptrs, hs, ws, n, wp), "pxr_set_image_prompts_sized")
        self._n_img = n
        self.n_prompts = [t_ + n for t_ in self._n_text]

    def set_spot_mask(self, mask):
        """fetch_spot_indexes (pixray.py:370-394): bool / 0-1 array [3, cut_size, cut_size] (or [cut_size, cut_size]), True
        where the resized mask image is >= 0.5."""
        m = np.asarray(mask.cpu() if torch.is_tensor(mask) else mask)
        if m.ndim == 2:
            m = np.broadcast_to(m[None], (3,) + m.shape)
        m = np.ascontiguousarray((m != 0).astype(np.uint8).reshape(3, self.cut_size, self.cut_size))
        self._check(self.lib.pxr_set_spot_mask(self.h, m.ctypes.data_as(C.c_void_p)), "pxr_set_spot_mask")

    def set_spot_prompts(self, clip_idx, which, embeds, weights, stops):
        """args.spot_prompts (which = 1) / args.spot_prompts_off (which = 0) of one perceptor (pixray.py:917-931): scored on
        the cutouts of the masked image, ahead of the regular prompts in the loss vector.  Empty list clears."""
        w = np.ascontiguousarray(np.asarray(weights, dtype=np.float32).reshape(-1))
        n = int(w.size)
        s = np.maximum(np.ascontiguousarray(np.asarray(stops, dtype=np.float32).reshape(-1)), np.float32(-3.0e38))
        D = self.clip_dims[clip_idx]
        e = np.ascontiguousarray(np.asarray(embeds, dtype=np.float32).reshape(n, D)) if n else np.zeros((1, D), np.float32)
        rc = self.lib.pxr_set_spot_prompts(self.h, clip_idx, int(which), e.ctypes.data_as(C.c_void_p), n, D,
                                           w.ctypes.data_as(C.c_void_p), s.ctypes.data_as(C.c_void_p))
        self._check(rc, "pxr_set_spot_prompts")
        self._n_spot[clip_idx][int(which)] = n

    def add_aux_loss(self, kind, weight, params):
        """One more entry of the loss vector / term of the gradient (pxr_add_aux_loss; Losses/*.py).  Returns the
        index of its value in the loss vector."""
        a = np.ascontiguousarray(np.asarray(params, dtype=np.float32).reshape(-1))
        rc = self.lib.pxr_add_aux_loss(self.h, int(kind), C.c_float(float(weight)), a.ctypes.data_as(C.c_void_p), int(a.size))
        self._check(rc, "pxr_add_aux_loss")
        return self.num_losses() - 1

    def add_filter(self, kind, weight, params):
        """One more filter between synth and the cutouts (pxr_add_filter; filters/*.py).  Its loss takes the next entry at the
        FRONT of the loss vector.  Returns the filter's index."""
        a = np.ascontiguousarray(np.asarray(params, dtype=np.float32).reshape(-1))
        rc = self.lib.pxr_add_filter(self.h, int(kind), C.c_float(float(weight)), a.ctypes.data_as(C.c_void_p), int(a.size))
        self._check(rc, "pxr_add_filter")
        self._n_filters = getattr(self, "_n_filters", 0) + 1
        return self._n_filters - 1

    def clear_filters(self):
        self._check(self.lib.pxr_clear_filters(self.h), "pxr_clear_filters")
        self._n_filters = 0

    def set_filter_shifts(self, filter_idx, rand_h, rand_w):
        """Fix one filter's (rand_h, rand_w) draws (replays / parity tests); negative values hand them back to the engine."""
        self._check(self.lib.pxr_set_filter_shifts(self.h, int(filter_idx), int(rand_h), int(rand_w)), "pxr_set_filter_shifts")

    def add_anchor(self, kind, weight, ref):
        """One anchor term between the latent (or the image, ANCHOR_PIX) and a stored copy (pxr_add_anchor; the init_weight
        family and image_labels, pixray.py:1344-1375).  `ref`: torch tensor (any device) or array; copied."""
        if torch.is_tensor(ref):
            r = ref.detach().to(torch.float32).contiguous()
            ptr, n, keep = C.c_void_p(r.data_ptr()), r.numel(), r
        else:
            keep = np.ascontiguousarray(np.asarray(ref, dtype=np.float32).reshape(-1))
            ptr, n = keep.ctypes.data_as(C.c_void_p), keep.size
        rc = self.lib.pxr_add_anchor(self.h, int(kind), C.c_float(float(weight)), ptr, C.c_longlong(int(n)))
        self._check(rc, "pxr_add_anchor")
        del keep

    def clear_anchors(self):
        self._check(self.lib.pxr_clear_anchors(self.h), "pxr_clear_anchors")

    def clear_aux_losses(self):
        self._check(self.lib.pxr_clear_aux_losses(self.h), "pxr_clear_aux_losses")

    def num_losses(self):
        n = C.c_int()
        self.lib.pxr_num_losses(self.h, C.byref(n))
        return n.value

    def read_losses(self):
        """The loss vector of the last forward/backward: prompts of every perceptor, then the auxiliary losses."""
        out = np.zeros(max(self.num_losses(), 1), dtype=np.float32)
        self._check(self.lib.pxr_read_losses(self.h, out.ctypes.data_as(C.c_void_p)), "pxr_read_losses")
        return out[:self.num_losses()]

    # ------------------------------------------------------------------ vdiff drawer
    def vdiff_set_schedule(self, steps, alphas, sigmas):
        """sample_state's steps / alphas / sigmas (vdiff.py:113-126, sampling.py:41-51)."""
        a = [np.ascontiguousarray(np.asarray(v, dtype=np.float32).reshape(-1)) for v in (steps, alphas, sigmas)]
        rc = self.lib.pxr_vdiff_set_schedule(self.h, *(v.ctypes.data_as(C.c_void_p) for v in a), int(a[0].size))
        self._check(rc, "pxr_vdiff_set_schedule")

    def vdiff_set_clip_embed(self, embed):
        e = np.ascontiguousarray(np.asarray(embed, dtype=np.float32).reshape(-1))
        self._check(self.lib.pxr_vdiff_set_clip_embed(self.h, e.ctypes.data_as(C.c_void_p), int(e.size)), "pxr_vdiff_set_clip_embed")

    def vdiff_set_iteration(self, i):
        self.lib.pxr_vdiff_set_iteration(self.h, int(i))

    def vdiff_renoise(self, z, i, noise=None):
        """drawer.makenoise(cur_it) (vdiff.py:156-157): in place on z; noise [1,3,H,W] ~ N(0,1) or None (eta = 0)."""
        if noise is not None:
            noise = noise.to(self.device, torch.float32).contiguous()
            torch.cuda.current_stream().synchronize()
        rc = self.lib.pxr_vdiff_renoise(self.h, self._p_inplace(z, "z"), int(i), self._p(noise))
        self._check(rc, "pxr_vdiff_renoise")
        self.sync()
        return z

    def init_comm(self):
        """Cutout-sharded multi-GPU mode: rank 0 draws an ncclUniqueId, torch.distributed (already initialised by the
        launcher) broadcasts it, and the engine builds its own communicator (pxr_set_comm)."""
        import os

        import torch.distributed as dist
        if self.world == 1:
            return
        if "PXR_NCCL_LIB" not in os.environ:
            try:
                import nvidia.nccl
                cand = os.path.join(os.path.dirname(nvidia.nccl.__file__), "lib", "libnccl.so.2")
                if os.path.exists(cand):
                    os.environ["PXR_NCCL_LIB"] = cand
            except Exception:
                pass
        buf = (C.c_ubyte * 128)()
        if self.rank == 0:
            rc = self.lib.pxr_get_unique_id(buf)
            if rc != 0:
                raise EngineError(f"pxr_get_unique_id failed ({rc}): {self.lib.pxr_last_error(None).decode()}")
        dev = self.device if dist.get_backend() == "nccl" else torch.device("cpu")
        t = torch.tensor(list(buf), dtype=torch.uint8, device=dev)
        dist.broadcast(t, src=0)
        raw = bytes(t.cpu().tolist())
        self._check(self.lib.pxr_set_comm(self.h, raw, self.rank, self.world), "pxr_set_comm")

    def z_bounds(self):
        zc = self.z_shape[1]
        lo, hi = self._new(zc), self._new(zc)
        self._check(self.lib.pxr_z_bounds(self.h, self._p(lo), self._p(hi)), "pxr_z_bounds")
        self.sync()
        return lo, hi

    def set_color_jitter(self, p=0.8, saturation=0.1, hue=0.1):
        """Distribution of the engine-drawn K.ColorJitter stage (pixray.py:416, 436); p=0 turns it off."""
        self._check(self.lib.pxr_set_color_jitter(self.h, C.c_float(p), C.c_float(saturation), C.c_float(hue)),
                    "pxr_set_color_jitter")

    def _cut_params(self, transforms, zoom_padding, fill, noise_facs, noise, color_jitter=None):
        p = _lib.CutParams()
        keep = []
        if color_jitter is not None:
            cj = np.ascontiguousarray(np.asarray(color_jitter, dtype=np.float32).reshape(self.cutn, 3))
            keep.append(cj)
            p.color_jitter = cj.ctypes.data_as(C.c_void_p)
        if transforms is not None:
            t = np.ascontiguousarray(np.asarray(transforms, dtype=np.float32).reshape(self.cutn, 9))
            keep.append(t)
            p.transforms = t.ctypes.data_as(C.c_void_p)
        p.zoom_padding, p.fill = int(zoom_padding), float(fill)
        if noise_facs is not None:
            f = np.ascontiguousarray(np.asarray(noise_facs, dtype=np.float32).reshape(self.cutn))
            keep.append(f)
            p.noise_facs = f.ctypes.data_as(C.c_void_p)
        if noise is not None:
            nz = noise.to(self.device, torch.float32).contiguous()
            keep.append(nz)
            p.noise = C.c_void_p(nz.data_ptr())
        self._keep = keep
        return p

    # ------------------------------------------------------------------ per-op entry points (parity tests)
    def synth(self, z):
        z = z.to(self.device, torch.float32).contiguous()
        out = self._new(1, 3, *self.image_hw)
        torch.cuda.current_stream().synchronize()
        self._check(self.lib.pxr_synth(self.h, self._p(z), self._p(out)), "pxr_synth")
        self.sync()
        return out

    def vqgan_encode(self, img):
        """z = model.encode(img)[0] (vqgan.py:174-185): img [1, 3, H, W] in [-1, 1] -> z [1, C, h, w] (codebook rows)."""
        img = img.to(self.device, torch.float32).reshape(1, 3, *self.image_hw).contiguous()
        out = self._new(*self.z_shape)
        torch.cuda.current_stream().synchronize()
        self._check(self.lib.pxr_vqgan_encode(self.h, self._p(img), self._p(out)), "pxr_vqgan_encode")
        self.sync()
        return out

    def make_cutouts(self, img=None, *, transforms=None, zoom_padding=PAD_REFLECTION, fill=0.0, noise_facs=None,
                     noise=None, it=0, use_engine_rng=False, color_jitter=None):
        if img is not None:
            img = img.to(self.device, torch.float32).contiguous()
        out = self._new(self.n_local, 3, self.cut_size, self.cut_size)
        p = None if use_engine_rng else self._cut_params(transforms, zoom_padding, fill, noise_facs, noise,
                                                                color_jitter)
        torch.cuda.current_stream().synchronize()
        rc = self.lib.pxr_make_cutouts(self.h, self._p(img), None if p is None else C.byref(p), it, self._p(out))
        self._check(rc, "pxr_make_cutouts")
        self.sync()
        return out

    def encode_image(self, clip_idx=0, batch=None):
        """Unit-norm embeddings of the engine's current cutouts, or of `batch` [cutn_local,3,cs,cs] when given."""
        out = self._new(self.n_local, self.clip_dims[clip_idx])
        if batch is not None:
            batch = batch.to(self.device, torch.float32).contiguous()
            torch.cuda.current_stream().synchronize()
        self._check(self.lib.pxr_encode_image(self.h, clip_idx, self._p(batch), self._p(out)), "pxr_encode_image")
        self.sync()
        return out

    def prompt_loss(self, clip_idx=0, embeds=None):
        if embeds is not None:
            embeds = embeds.to(self.device, torch.float32).contiguous()
            torch.cuda.current_stream().synchronize()
        out = self._new(self.n_prompts[clip_idx])
        self._check(self.lib.pxr_prompt_loss(self.h, clip_idx, self._p(embeds), self._p(out)), "pxr_prompt_loss")
        self.sync()
        return out

    def backward(self):
        g = self._new(*self.z_shape)
        self._check(self.lib.pxr_backward(self.h, self._p(g)), "pxr_backward")
        self.sync()
        return g

    def step(self, z, lr, it=0):
        self._check(self.lib.pxr_step(self.h, self._p_inplace(z, "z"), C.c_float(lr), it), "pxr_step")
        self.sync()
        return z

    def reset_optimizer(self):
        """A fresh instance of the current optimiser: state zeroed, step count 0 (pxr_reset_optimizer)."""
        self._check(self.lib.pxr_reset_optimizer(self.h), "pxr_reset_optimizer")

    def set_optimizer(self, name):
        """Switch to the optimiser `name` (a key of OPTIMISERS) with fresh state (pxr_set_optimizer)."""
        if name not in OPTIMISERS:
            raise NotImplementedError(f"optimiser '{name}' is not built; available: {sorted(OPTIMISERS)}")
        self._check(self.lib.pxr_set_optimizer(self.h, OPTIMISERS[name]), "pxr_set_optimizer")
        self.optimizer = name

    def save_state(self):
        """bytes: z, the optimiser's state / kind / step and the drop bookkeeping (pxr_save_state)."""
        n = C.c_int64()
        self.lib.pxr_state_size(self.h, C.byref(n))
        buf = (C.c_ubyte * n.value)()
        self._check(self.lib.pxr_save_state(self.h, buf), "pxr_save_state")
        return bytes(buf)

    def load_state(self, blob):
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        self._check(self.lib.pxr_load_state(self.h, buf), "pxr_load_state")

    def read_z(self):
        """The engine's current latent (a copy)."""
        return self.debug_read("z", self.z_shape)

    def set_z_grad(self, g):
        """The gradient the next step() applies (the plugin loop accumulates z.grad over several passes itself)."""
        self._check(self.lib.pxr_set_z_grad(self.h, self._p_inplace(g, "z.grad")), "pxr_set_z_grad")

    def set_batches(self, batches):
        """args.batches (pixray.py:1464-1482): passes per iterate(), gradients accumulated, one optimiser step."""
        self._check(self.lib.pxr_set_batches(self.h, int(batches)), "pxr_set_batches")

    def set_schedule(self, base_lr, iter_drop_delay=12, max_loss_drops=0, auto_stop=False, drops=()):
        """checkdrop / learning-rate drops / auto-stop on the device (pxr_set_schedule): iterate() then ignores `lr`."""
        d = np.ascontiguousarray(np.asarray(list(drops), dtype=np.int32).reshape(-1))
        self._check(self.lib.pxr_set_schedule(self.h, C.c_float(float(base_lr)), int(iter_drop_delay), int(max_loss_drops),
                                              int(bool(auto_stop)), d.ctypes.data_as(C.c_void_p), int(d.size)),
                    "pxr_set_schedule")

    def poll_status(self):
        """The last completed managed iteration's record, read from pinned memory WITHOUT synchronising; None when no
        consistent record is available yet."""
        st = _lib.Status()
        rc = self.lib.pxr_poll_status(self.h, C.byref(st))
        if rc != 0:
            return None
        return dict(iter=st.iter, loss_sum=st.loss_sum, best_loss=st.best_loss, best_iter=st.best_iter,
                    num_loss_drop=st.num_loss_drop, stopped=bool(st.stopped), rebuilt=bool(st.rebuilt), lr=st.lr,
                    losses=np.array(st.losses[:st.n_losses], dtype=np.float32))

    # ------------------------------------------------------------------ the fast path (what bench.py times)
    def iterate(self, z, lr, it, *, params=None, losses_out=None):
        """One train() iteration entirely inside the library.  params: dict(transforms, zoom_padding, fill,
        noise_facs, noise, color_jitter) or None for the engine's own Philox draws.  losses_out: float32 numpy array (host) to
        receive the per-prompt losses (forces a stream sync), or None."""
        p = None
        if params is not None:
            p = self._cut_params(params.get("transforms"), params.get("zoom_padding", it % 2),
                                 params.get("fill", 0.0), params.get("noise_facs"), params.get("noise"),
                                 params.get("color_jitter"))
        # z / noise may have been produced on torch's stream (e.g. an H2D copy still in flight): order the engine's
        # non-blocking stream after it without a host sync
        if self._ext is None:
            self._ext = torch.cuda.ExternalStream(self.stream_ptr())
        self._ext.wait_stream(torch.cuda.current_stream())
        lp = None if losses_out is None else losses_out.ctypes.data_as(C.c_void_p)
        rc = self.lib.pxr_iterate(self.h, self._p_inplace(z, "z"), C.c_float(lr), it, None if p is None else C.byref(p), lp)
        self._check(rc, "pxr_iterate")

    def debug_read(self, name, shape, dtype=torch.float32):
        out = torch.empty(*shape, device=self.device, dtype=dtype)
        rc = self.lib.pxr_debug_read(self.h, name.encode(), self._p(out), C.c_int64(out.numel() * out.element_size()))
        self._check(rc, f"pxr_debug_read({name})")
        return out

    def profile_iteration(self, z, lr, it):
        out = (C.c_double * 6)()
        tb = C.c_double(0.0)
        self._check(self.lib.pxr_profile_iteration2(self.h, self._p_inplace(z, "z"), C.c_float(lr), it, out, C.byref(tb)),
                    "pxr_profile_iteration2")
        return dict(gemm_ms=out[0], gemm_launches=int(out[1]), gemm_flops=out[2], other_ms=out[3],
                    other_launches=int(out[4]), total_ms=out[5], gemm_bytes=tb.value)

    def stream_ptr(self):
        p = C.c_void_p()
        self.lib.pxr_get_stream(self.h, C.byref(p))
        return p.value

    def num_launches(self):
        n = C.c_int64()
        self.lib.pxr_num_kernel_launches(self.h, C.byref(n))
        return n.value
