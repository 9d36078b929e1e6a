"""Mirror of the hot-path pieces of the reference's ``diffhandles/guided_stable_diffuser.py``:
``get_depth_intrinsics`` (:129-153), ``process_correspondences`` (:490-584) and the guidance weight
schedules (:336-373, :612-665).  The U-Net, VAE, text encoder and scheduler stay stock PyTorch/diffusers and
are outside this build (north star), so ``GuidedStableDiffuser`` here carries no model weights.
"""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch

from . import _native as N
from .utils import unpack_correspondences

LATENT_GRID = 64   # guided_stable_diffuser.py:526-529: the loss grid is hard-wired to 64 x 64


class ProcessedCorrespondences(dict):
    """The reference's dict of ten NumPy int64 index arrays, plus the device-side int32 cell lists the CUDA
    loss kernels consume (``.device_lists``), so no index array is re-uploaded per loss call."""
    device_lists: Dict[str, torch.Tensor]
    grid: int


def process_correspondences_device(corr: torch.Tensor, img_res: int, bg_erosion: int = 0, grid: int = LATENT_GRID,
                                   device: torch.device = None) -> ProcessedCorrespondences:
    """corr (N,4) int64 (CPU or CUDA).  One kernel launch + one small device->host copy."""
    lib = N.load()
    if device is None:
        device = corr.device if corr.is_cuda else torch.device("cuda", torch.cuda.current_device())
    c = corr.to(device=device, dtype=torch.int64).reshape(-1, 4).contiguous()
    n = c.shape[0]
    cells = grid * grid
    i32 = torch.int32
    fg_src = torch.empty(max(n, 1), dtype=i32, device=device)
    fg_dst = torch.empty(max(n, 1), dtype=i32, device=device)
    bg = torch.empty(cells, dtype=i32, device=device)
    bg_o = torch.empty(cells, dtype=i32, device=device)
    bg_t = torch.empty(cells, dtype=i32, device=device)
    counts = torch.zeros(8, dtype=i32, device=device)
    N.check(lib.dh_process_correspondences(N.ptr(c) if n else None, n, int(img_res), grid, int(bg_erosion), N.ptr(fg_src),
                                           N.ptr(fg_dst), N.ptr(bg), N.ptr(bg_o), N.ptr(bg_t), N.ptr(counts),
                                           N.stream_handle(device)), "dh_process_correspondences")
    nv, nb, nbo, nbt = counts[:4].tolist()
    dl = {"fg_src": fg_src[:nv], "fg_dst": fg_dst[:nv], "bg": bg[:nb], "bg_orig": bg_o[:nbo], "bg_trans": bg_t[:nbt]}
    host = {k: v.cpu().numpy().astype(np.int64) for k, v in dl.items()}
    pc = ProcessedCorrespondences({
        'original_x': host["fg_src"] % grid, 'original_y': host["fg_src"] // grid,
        'transformed_x': host["fg_dst"] % grid, 'transformed_y': host["fg_dst"] // grid,
        'background_x': host["bg"] % grid, 'background_y': host["bg"] // grid,
        'background_x_orig': host["bg_orig"] % grid, 'background_y_orig': host["bg_orig"] // grid,
        'background_x_trans': host["bg_trans"] % grid, 'background_y_trans': host["bg_trans"] // grid,
    })
    pc.device_lists = dl
    pc.grid = grid
    return pc


class GuidanceWeightSchedule:
    """Base schedule (guided_stable_diffuser.py:612-620): unit weights for the three guided layers at every step."""

    def __call__(self, denoising_step: int, optimization_step: int):
        return [1.0, 1.0, 1.0], [1.0, 1.0, 1.0]


class _StepTable:
    """Piecewise-constant weight table: rows (first_step, fg_weights, bg_weights); a step uses the row with the largest
    first_step that does not exceed it."""

    def __init__(self, rows, what: str):
        rows = sorted(rows, key=lambda r: r[0])
        for _, fg, bg in rows:
            if len(fg) != len(bg):
                raise ValueError("Number of foreground and background weights do not match.")
        self.what = what
        self.starts = [r[0] for r in rows]
        self.weights = [(list(r[1]), list(r[2])) for r in rows]
        self.width = len(rows[0][1])

    def at(self, step: int):
        import bisect
        i = bisect.bisect_right(self.starts, step) - 1
        return self.weights[i] if i >= 0 else None


class StepGuidanceWeightSchedule(GuidanceWeightSchedule):
    """guided_stable_diffuser.py:622-665: per-layer weights = (weights of the denoising step) x (weights of the optimisation
    iteration), each looked up in a piecewise-constant table.  Same constructor arguments and errors as the reference."""

    def __init__(self, denoising_steps, optimization_steps):
        self._denoising = _StepTable(denoising_steps, "denoising")
        self._optimization = _StepTable(optimization_steps, "optimization")
        if self._denoising.width != self._optimization.width:
            raise ValueError("Number of denoising and optimization weights do not match.")
        self.denoising_steps = list(zip(self._denoising.starts, *zip(*self._denoising.weights)))
        self.optimization_steps = list(zip(self._optimization.starts, *zip(*self._optimization.weights)))

    def __call__(self, denoising_step: int, optimization_step: int):
        den, opt = self._denoising.at(denoising_step), self._optimization.at(optimization_step)
        if den is None or opt is None:
            raise ValueError(f"Could not find weights for denoising step {denoising_step} and optimization step {optimization_step}.")
        return [d * o for d, o in zip(den[0], opt[0])], [d * o for d, o in zip(den[1], opt[1])]


# guided_stable_diffuser.py:336-373 - which of the three guided layers is active in denoising step t (t mod 3), and the
# multipliers of the optimisation iterations 0..3
_LAYER_PATTERN = (((0.0, 0.0, 7.5), (0.0, 0.0, 1.5)),
                  ((0.0, 5.0, 0.0), (0.0, 1.5, 0.0)),
                  ((0.0, 5.0, 7.5), (0.0, 1.5, 1.5)))
_ITERATION_GAIN = ((2.5, 1.25), (1.25, 2.5), (1.25, 1.25), (2.5, 2.5))


def _fade(weight: float, steps: int, kind: str) -> np.ndarray:
    """Weight over the guided denoising steps: constant, linear to zero, or quadratic to zero (np.linspace like the reference)."""
    if kind == "constant":
        return np.linspace(weight, weight, steps)
    if kind == "linear":
        return np.linspace(weight, 0.0, steps)
    if kind == "quadratic":
        return np.linspace(np.sqrt(weight), 0.0, steps) ** 2
    raise ValueError(f"Unknown guidance schedule type: {kind}")


def make_guidance_weight_schedule(fg_weight: float, bg_weight: float, guidance_max_step: int = 38,
                                  guidance_schedule_type: str = "constant") -> StepGuidanceWeightSchedule:
    """The schedule ``guided_inference`` builds (guided_stable_diffuser.py:336-373): user weights x 30, faded over the first
    ``guidance_max_step`` denoising steps, distributed over the layers by ``t mod 3``, zero afterwards."""
    fg_fade = _fade(fg_weight * 30, guidance_max_step, guidance_schedule_type)
    bg_fade = _fade(bg_weight * 30, guidance_max_step, guidance_schedule_type)
    denoising = []
    for t in range(guidance_max_step):
        fg_pat, bg_pat = _LAYER_PATTERN[t % 3]
        denoising.append((t, (np.array(fg_pat) * fg_fade[t]).tolist(), (np.array(bg_pat) * bg_fade[t]).tolist()))
    denoising.append((guidance_max_step, [0.0] * 3, [0.0] * 3))
    optimization = [(i, [f] * 3, [b] * 3) for i, (f, b) in enumerate(_ITERATION_GAIN)]
    return StepGuidanceWeightSchedule(denoising_steps=denoising, optimization_steps=optimization)


class GuidedStableDiffuser:
    """The reference class's hot-path methods under their own names and signatures.  The diffusion models themselves
    (U-Net with recorded activations, VAE, CLIP tokenizer / text encoder, DDIM scheduler) are stock PyTorch / diffusers
    objects outside this build: pass them in (``unet=..., scheduler=..., vae=..., tokenizer=..., text_encoder=...``) and
    ``guided_inference`` runs the reference's guided denoising loop with the fused sm_100a loss kernel in it."""

    def __init__(self, conf=None, unet=None, scheduler=None, vae=None, tokenizer=None, text_encoder=None):
        self.conf = conf
        self.unet, self.scheduler, self.vae, self.tokenizer, self.text_encoder = unet, scheduler, vae, tokenizer, text_encoder
        self.device = torch.device("cpu")

    def to(self, device: torch.device = None):
        for m in (self.unet, self.vae, self.text_encoder):
            if m is not None and hasattr(m, "to"):
                m.to(device=device)
        self.device = device
        return self

    def _conf(self, name, default):
        return getattr(self.conf, name, default) if self.conf is not None else default

    def get_feature_shape(self):
        """guided_stable_diffuser.py:104-109: latent grid of the injected U-Net (64 x 64 x 4 for SD2-depth)."""
        cfg = getattr(self.unet, "config", None)
        n = int(getattr(cfg, "sample_size", LATENT_GRID)) if cfg is not None else LATENT_GRID
        return [n, n, 4]

    def init_depth(self, depth):
        """guided_stable_diffuser.py:111-127: bicubic resize to the latent grid, then min/max normalisation to [-1, 1]."""
        h, w = self.get_feature_shape()[:2]
        depth = torch.nn.functional.interpolate(depth, size=(h, w), mode="bicubic", align_corners=False)
        lo = torch.amin(depth, dim=[1, 2, 3], keepdim=True)
        hi = torch.amax(depth, dim=[1, 2, 3], keepdim=True)
        return 2.0 * (depth - lo) / (hi - lo) - 1.0

    def get_image_shape(self):
        """guided_stable_diffuser.py:82-85: feature shape times the VAE's down-scaling factor."""
        h, w = self.get_feature_shape()[:2]
        f = 2 ** (len(self.vae.config.block_out_channels) - 1) if self.vae is not None else 8
        return (h * f, w * f, 3)

    def prepare_extra_step_kwargs(self, generator, eta):
        """guided_stable_diffuser.py:595-610: ``eta`` / ``generator`` only for schedulers whose ``step`` accepts them."""
        import inspect
        accepted = set(inspect.signature(self.scheduler.step).parameters.keys())
        extra = {}
        if "eta" in accepted:
            extra["eta"] = eta
        if "generator" in accepted:
            extra["generator"] = generator
        return extra

    def encode_latent_image(self, image: torch.Tensor) -> torch.Tensor:
        """guided_stable_diffuser.py:277-283: not implemented by the reference either."""
        raise NotImplementedError

    def get_timesteps(self, num_inference_steps, strength):
        """guided_stable_diffuser.py:586-593."""
        init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
        t_start = max(num_inference_steps - init_timestep, 0)
        return self.scheduler.timesteps[t_start * getattr(self.scheduler, "order", 1):], num_inference_steps - t_start

    def guided_inference(self, latents: torch.Tensor, depth: torch.Tensor, uncond_embeddings: torch.Tensor, prompt: str,
                         activations_orig, correspondences: torch.Tensor, fg_weight: float = None, bg_weight: float = None,
                         save_denoising_steps: bool = False):
        """guided_stable_diffuser.py:291-488, same signature.  Per denoising step up to ``num_optsteps`` gradient steps on
        the latents driven by sum_l fgw[l] L_fg,l + bgw[l] L_bg,l (ONE fused K4 launch per evaluation, :415-434), then the
        classifier-free-guidance forward (scale 7.5, :452-470) and the scheduler step; finally the VAE decode.  Needs the
        injected diffusion models; without them this raises NotImplementedError (they are outside this build)."""
        return self._guided_inference(False, latents, depth, uncond_embeddings, prompt, activations_orig, correspondences, fg_weight,
                                      bg_weight, save_denoising_steps)

    def guided_inference_batch(self, latents: torch.Tensor, depth: torch.Tensor, uncond_embeddings, prompt,
                               activations_orig, correspondences, fg_weight: float = None, bg_weight: float = None):
        """``guided_inference`` for B edits at once (``guided_denoise_batch``): the U-Net runs at batch B, each guided step
        evaluates the losses of all edits in one K4 launch.  ``depth`` is (B,1,H,W), ``correspondences`` a list of B (N,4)
        lists; ``latents`` (1,4,h,w) is shared by every edit, or (B,4,h,w); ``activations_orig`` is one identity shared by every
        edit, or a list of B identities.  ``prompt`` is one prompt (string or embedding) shared by every edit, a list of B
        strings or a (B,L,D) embedding; ``uncond_embeddings`` is one null-text sequence shared by every edit or a list of B
        sequences, so edits of different images run in one batch.  Returns the B decoded images.  The saved denoising steps of
        ``save_denoising_steps`` are not supported here."""
        return self._guided_inference(True, latents, depth, uncond_embeddings, prompt, activations_orig, correspondences, fg_weight,
                                      bg_weight, False)

    def _guided_inference(self, batch, latents, depth, uncond_embeddings, prompt, activations_orig, correspondences, fg_weight,
                          bg_weight, save_denoising_steps):
        """The body of ``guided_inference`` (batch=False: one edit, ``guided_denoise``) and ``guided_inference_batch``
        (batch=True: B edits, ``guided_denoise_batch``)."""
        from .guided_loop import guided_denoise, guided_denoise_batch
        name = "guided_inference_batch" if batch else "guided_inference"
        missing = [n for n in ("unet", "scheduler") if getattr(self, n) is None]
        if missing:
            raise NotImplementedError(f"{name} needs the stock diffusion models ({', '.join(missing)}); pass them to "
                                      "GuidedStableDiffuser(conf, unet=..., scheduler=..., vae=..., tokenizer=..., text_encoder=...)")
        corrs = correspondences if batch else [correspondences]
        B = len(corrs)
        if batch:
            if self._conf("save_denoising_steps", False):
                raise NotImplementedError("guided_inference_batch does not save the denoising steps; use guided_inference per edit")
            if depth.shape[0] != B:
                raise ValueError(f"depth must be (B,1,H,W) with B = {B} edits, got {tuple(depth.shape)}")
            if latents.shape[0] not in (1, B):
                raise ValueError(f"latents must be (1,4,h,w) or ({B},4,h,w), got {tuple(latents.shape)}")
            if isinstance(uncond_embeddings, (list, tuple)) and len(uncond_embeddings) != B:
                raise ValueError(f"uncond_embeddings must be one sequence or a list of B = {B} sequences, got {len(uncond_embeddings)}")
            if isinstance(prompt, (list, tuple)) and len(prompt) != B:
                raise ValueError(f"prompt must be one prompt or a list of B = {B} prompts, got {len(prompt)}")
        fg_weight = self._conf("fg_weight", 1.5) if fg_weight is None else fg_weight
        bg_weight = self._conf("bg_weight", 1.25) if bg_weight is None else bg_weight
        use_depth = self._conf("use_depth", True)
        with torch.no_grad():
            generator = torch.manual_seed(self._conf("seed", 2773))
            n_steps = self._conf("num_timesteps", 50)
            self.scheduler.set_timesteps(n_steps, device=self.device)
            timesteps, _ = self.get_timesteps(n_steps, 1.0)
            pcs = [self.process_correspondences(c, img_res=depth.shape[-1], bg_erosion=self._conf("bg_erosion", 0)) for c in corrs]
            if use_depth:
                depth = self.init_depth(depth)
            if batch and isinstance(prompt, (list, tuple)):
                cond = torch.cat([self._encode_prompt(p) for p in prompt])
            else:
                cond = self._encode_prompt(prompt)
            extra = self.prepare_extra_step_kwargs(generator, 0.0)
            if batch:
                if cond.shape[0] not in (1, B):
                    raise ValueError(f"the prompt embedding must be (1,L,D) or ({B},L,D), got {tuple(cond.shape)}")
                cond = cond.expand(B, *cond.shape[1:])
                latents = latents.expand(B, *latents.shape[1:]).contiguous()

        def uncond_at(t_idx):
            """the null-text embedding of step t_idx: shared, or each edit's own stacked to (B,L,D)"""
            if batch and isinstance(uncond_embeddings, (list, tuple)):
                return torch.cat([u[t_idx].expand(1, *cond.shape[1:]) for u in uncond_embeddings])
            return uncond_embeddings[t_idx]

        def unet_fn(model_in, t):
            if use_depth:
                model_in = torch.cat([model_in, depth], dim=1)
            out = self.unet(model_in, t, encoder_hidden_states=cond, cross_attention_kwargs=None, return_dict=False)
            return out[0], [out[4], out[5], out[6]]

        def cfg_pair(lat, t, t_idx):
            return self._cfg_forward(lat, t, uncond_at(t_idx), cond, depth if use_depth else None)

        def cfg_noise(lat, t, t_idx):
            n_uncond, n_text = cfg_pair(lat, t, t_idx)
            return n_uncond + 7.5 * (n_text - n_uncond)

        # a diffusers DDIMScheduler (epsilon prediction, eta = 0, no clipping: the reference's, :31-32) is replaced by the fused
        # CFG + DDIM update; any other scheduler object keeps its own step()
        ddim = self._fused_ddim()

        steps = {'opt': [], 'post-opt': []} if save_denoising_steps else None

        def on_step(kind, lat):
            if kind == 'opt':
                steps['opt'].append([self.decode_latent_image(lat.detach()).cpu()])
            else:
                steps['opt'][-1].append(self.decode_latent_image(lat.detach()).cpu())

        denoise = guided_denoise_batch if batch else guided_denoise
        latents = denoise(
            latents, timesteps, unet_fn, lambda noise, t, lat: self.scheduler.step(noise, t, lat, **extra, return_dict=False)[0],
            activations_orig, pcs if batch else pcs[0], fg_weight=fg_weight, bg_weight=bg_weight, num_optsteps=self._conf("num_optsteps", 3),
            guidance_max_step=self._conf("guidance_max_step", 38), guidance_schedule_type=self._conf("guidance_schedule_type", "constant"),
            bg_loss_type=self._conf("bg_loss_type", "global_avg"), fg_patch_size=self._conf("fg_patch_size", 1),
            bg_patch_size=self._conf("bg_patch_size", 1), scale_model_input=self.scheduler.scale_model_input, cfg_noise=cfg_noise,
            on_step=on_step if steps is not None else None, ddim=ddim, cfg_pair=cfg_pair if ddim is not None else None,
            # the schedule gives layer 0 the weight 0 at every step (:352-360): 0 * loss adds nothing to the value or to the latent
            # gradient, so such layers are not sent to the loss kernel (17 instead of 42 us per evaluation for SD2-depth)
            skip_zero_weight_layers=True)
        with torch.no_grad():
            image = self.decode_latent_image(latents)
        return (image, steps) if save_denoising_steps else image

    def _fused_ddim(self):
        """DDIMSchedule of the injected scheduler when the fused update reproduces its step(), else None."""
        from .guided_loop import DDIMSchedule
        if getattr(self.scheduler, "init_noise_sigma", 1.0) != 1.0:
            return None
        return DDIMSchedule.from_scheduler(self.scheduler)

    def _cfg_forward(self, latents, t, uncond_embedding, cond, depth):
        """The classifier-free-guidance forward (guided_stable_diffuser.py:243-263, :452-468): the latents twice, the
        unconditional and the prompt embedding -> (noise_uncond, noise_text)."""
        model_in = self.scheduler.scale_model_input(torch.cat([latents] * 2), t)
        if depth is not None:
            model_in = torch.cat([model_in, torch.cat([depth] * 2, dim=0)], dim=1)
        emb = torch.cat([uncond_embedding.expand(*cond.shape), cond])
        noise = self.unet(model_in, t, encoder_hidden_states=emb, cross_attention_kwargs=None, return_dict=False)[0]
        return noise.chunk(2)

    def _encode_prompt(self, prompt):
        if self.tokenizer is not None and self.text_encoder is not None and isinstance(prompt, str):
            ids = self.tokenizer([prompt], padding="max_length", truncation=True, max_length=self.tokenizer.model_max_length,
                                 return_tensors="pt")
            return self.text_encoder(ids.input_ids.to(self.device))[0]
        if isinstance(prompt, str):
            raise NotImplementedError("a prompt string needs the stock tokenizer / text encoder; pass them to GuidedStableDiffuser(...) "
                                      "or pass the prompt embedding instead of the string")
        return prompt                            # a pre-computed prompt embedding may be passed instead of a string

    def initial_inference(self, init_latents: torch.Tensor, depth: torch.Tensor, uncond_embeddings: torch.Tensor, prompt: str):
        """guided_stable_diffuser.py:155-274, same signature: the recording pass.  Per timestep one conditional U-Net forward whose
        three guided activations are written straight into pre-allocated device-resident (T,C,h,w) stacks (``ActivationRecorder``:
        no per-step list + final ``torch.stack`` copy of the 1.05 GB), then the classifier-free-guidance forward and the scheduler
        update (fused into one launch for a DDIM scheduler).  Returns (activations, latents, uncond_embeddings, init_latents).
        ``init_latents=None`` (fresh noise from the seeded generator, :192-200) needs ``scheduler.add_noise``."""
        from .identity import ActivationRecorder
        from .guided_loop import cfg_ddim_step
        missing = [n for n in ("unet", "scheduler") if getattr(self, n) is None]
        if missing:
            raise NotImplementedError(f"initial_inference needs the stock diffusion models ({', '.join(missing)}); pass them to "
                                      "GuidedStableDiffuser(conf, unet=..., scheduler=..., vae=..., tokenizer=..., text_encoder=...)")
        use_depth = self._conf("use_depth", True)
        with torch.no_grad():
            generator = torch.manual_seed(self._conf("seed", 2773))
            n_steps = self._conf("num_timesteps", 50)
            self.scheduler.set_timesteps(n_steps, device=self.device)
            timesteps, _ = self.get_timesteps(n_steps, 1.0)
            if use_depth:
                depth = self.init_depth(depth)
            cond = self._encode_prompt(prompt)
            if uncond_embeddings is None:
                uncond_embeddings = self._encode_prompt("")[[0]]
            if uncond_embeddings.shape[0] == 0:
                uncond_embeddings = uncond_embeddings.expand(len(timesteps), -1, -1, -1)
            if init_latents is None:
                cfg = self.unet.config
                ch = cfg.in_channels - 1 if use_depth else cfg.in_channels
                shape = [1, ch, cfg.sample_size, cfg.sample_size]
                noise = torch.randn(shape, generator=generator, dtype=torch.float32).to(self.device)
                init_latents = self.scheduler.add_noise(torch.zeros(shape, device=self.device, dtype=torch.float32), noise, timesteps[0])
            extra = self.prepare_extra_step_kwargs(generator, 0.0)
            ddim = self._fused_ddim()
            t_host = [int(v) for v in (timesteps.tolist() if isinstance(timesteps, torch.Tensor) else timesteps)] if ddim is not None else None
            recorder = ActivationRecorder(len(timesteps))
            latents = init_latents
            for t_idx, t in enumerate(timesteps):
                model_in = self.scheduler.scale_model_input(latents, t)
                if use_depth:
                    model_in = torch.cat([model_in, depth], dim=1)
                out = self.unet(model_in, t, encoder_hidden_states=cond, cross_attention_kwargs=None, return_dict=False)
                recorder.record(t_idx, [out[4][0], out[5][0], out[6][0]])
                uemb = uncond_embeddings[t_idx] if uncond_embeddings.shape[0] == len(timesteps) else uncond_embeddings[0]
                n_uncond, n_text = self._cfg_forward(latents, t, uemb, cond, depth if use_depth else None)
                if ddim is not None:
                    latents = cfg_ddim_step(n_uncond, n_text, latents, ddim.coefficients(t_host[t_idx], 7.5)).view(latents.shape)
                else:
                    latents = self.scheduler.step(n_uncond + 7.5 * (n_text - n_uncond), t, latents, **extra, return_dict=False)[0]
        return recorder.stacks(), latents, uncond_embeddings, init_latents

    def decode_latent_image(self, latent_image: torch.Tensor) -> torch.Tensor:
        """guided_stable_diffuser.py:285-288 (VAE decode + the [0,1] post-processing of diffusers' VaeImageProcessor)."""
        if self.vae is None:
            return latent_image
        image = self.vae.decode(latent_image / self.vae.config.scaling_factor, return_dict=False)[0]
        return (image / 2 + 0.5).clamp(0, 1)

    @staticmethod
    def get_depth_intrinsics(device: torch.device = None):
        """guided_stable_diffuser.py:129-153: 55 degree FoV pinhole, principal point 0, image plane [-1,1]^2."""
        fov = 55.0
        f = 1.0 / np.tan(0.5 * fov * (np.pi / 180.0))
        return torch.tensor([[f, 0, 0.0], [0, f, 0.0], [0, 0, 1]], dtype=torch.float32, device=device)

    def process_correspondences(self, correspondences, img_res, bg_erosion=0):
        """guided_stable_diffuser.py:490-584 - returns the reference's dict of NumPy int64 arrays (a dict
        subclass that also keeps the device-side lists for the loss kernels)."""
        ox, oy, tx, ty = unpack_correspondences(correspondences)   # keeps the reference's (N,4) contract
        del ox, oy, tx, ty
        return process_correspondences_device(correspondences, img_res, bg_erosion)
