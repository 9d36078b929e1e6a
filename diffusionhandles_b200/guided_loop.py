"""The guided denoising loop around the (stock PyTorch) U-Net - SURVEY.md 8(f) rank 4, mirroring
guided_stable_diffuser.py:377-480: per timestep up to ``num_optsteps`` gradient steps on the latents, driven by the
fused guidance loss (one K4 launch per evaluation instead of six loss calls), then the classifier-free-guidance step.
The elementwise work between the U-Net calls is one launch each: ``latent_step`` (latents -= 0.1 grad, :434) and
``cfg_ddim_step`` (CFG combine + DDIM update, :470-474), with the DDIM coefficients of ``DDIMSchedule``.

The U-Net, the scheduler and the text embeddings are injected as callables / tensors; this module contains no model.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _native as N
from .guided_stable_diffuser import make_guidance_weight_schedule
from .losses import guidance_loss, guidance_loss_and_grad, guidance_loss_and_grad_batch


class DDIMSchedule:
    """The coefficients of the DDIM scheduler the reference constructs (guided_stable_diffuser.py:31-32:
    ``DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
    set_alpha_to_one=False)``; diffusers 0.23 defaults otherwise: 1000 training timesteps, epsilon prediction, "leading"
    timestep spacing, steps_offset 0), computed with the same fp32 torch ops on the CPU, so that the values handed to
    ``dh_cfg_ddim_step`` are the 0-d tensors ``DDIMScheduler.step`` would multiply with."""

    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012,
                 beta_schedule: str = "scaled_linear", set_alpha_to_one: bool = False, steps_offset: int = 0,
                 alphas_cumprod: Optional[torch.Tensor] = None, final_alpha_cumprod=None):
        if alphas_cumprod is None:
            if beta_schedule == "scaled_linear":
                betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
            elif beta_schedule == "linear":
                betas = torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
            else:
                raise NotImplementedError(f"{beta_schedule} is not implemented for DDIMSchedule")
            alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)
        self.alphas_cumprod = alphas_cumprod.detach().to(device="cpu", dtype=torch.float32)
        self.num_train_timesteps = int(self.alphas_cumprod.numel())
        if final_alpha_cumprod is None:
            final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]
        self.final_alpha_cumprod = torch.as_tensor(final_alpha_cumprod).detach().to(device="cpu", dtype=torch.float32).reshape(())
        self.steps_offset = int(steps_offset)
        self.num_inference_steps: Optional[int] = None
        self.timesteps: Optional[np.ndarray] = None
        self._coeffs: Dict[tuple, N.dh_ddim_coeffs] = {}

    @classmethod
    def from_scheduler(cls, scheduler) -> Optional["DDIMSchedule"]:
        """A table for an injected diffusers ``DDIMScheduler`` (None when the object is not one the fused update reproduces:
        no ``alphas_cumprod`` / ``final_alpha_cumprod``, v-prediction, clipping or thresholding)."""
        a, f = getattr(scheduler, "alphas_cumprod", None), getattr(scheduler, "final_alpha_cumprod", None)
        cfg = getattr(scheduler, "config", None)
        if not isinstance(a, torch.Tensor) or f is None or cfg is None:
            return None
        get = cfg.get if isinstance(cfg, dict) else lambda k, d=None: getattr(cfg, k, d)
        if get("prediction_type", "epsilon") != "epsilon" or get("clip_sample", False) or get("thresholding", False):
            return None
        if get("timestep_spacing", "leading") != "leading":
            return None
        sch = cls(alphas_cumprod=a, final_alpha_cumprod=f, steps_offset=get("steps_offset", 0))
        if getattr(scheduler, "num_inference_steps", None):
            sch.set_timesteps(int(scheduler.num_inference_steps))
        return sch

    def set_timesteps(self, num_inference_steps: int) -> np.ndarray:
        """"leading" spacing: (arange(n) * (N // n)).round()[::-1] + steps_offset, as int64 (980, 960, ..., 0 for n = 50)."""
        if num_inference_steps > self.num_train_timesteps:
            raise ValueError("num_inference_steps cannot exceed the number of training timesteps")
        self.num_inference_steps = int(num_inference_steps)
        ratio = self.num_train_timesteps // self.num_inference_steps
        self.timesteps = (np.arange(0, num_inference_steps) * ratio).round()[::-1].copy().astype(np.int64) + self.steps_offset
        self._coeffs.clear()
        return self.timesteps

    def coefficients(self, timestep: int, guidance_scale: float = 7.5, divide_by_reciprocal: bool = True) -> N.dh_ddim_coeffs:
        """dh_ddim_coeffs of one update (DDIMScheduler.step with eta = 0): every value is produced by the fp32 tensor expression of
        the scheduler - ``alpha_prod_t ** 0.5``, ``(1 - alpha_prod_t) ** 0.5``, ``(1 - alpha_prod_t_prev - std_dev_t**2) ** 0.5``."""
        if self.num_inference_steps is None:
            raise RuntimeError("call set_timesteps first")
        key = (int(timestep), float(guidance_scale), bool(divide_by_reciprocal))
        c = self._coeffs.get(key)
        if c is None:
            t = int(timestep)
            if not 0 <= t < self.num_train_timesteps:
                raise IndexError(f"timestep {t} outside the {self.num_train_timesteps} training timesteps")
            prev = t - self.num_train_timesteps // self.num_inference_steps
            alpha_t = self.alphas_cumprod[t]
            alpha_prev = self.alphas_cumprod[prev] if prev >= 0 else self.final_alpha_cumprod
            beta_t = 1 - alpha_t
            beta_prev = 1 - alpha_prev
            variance = (beta_prev / beta_t) * (1 - alpha_t / alpha_prev)
            std_dev_t = 0.0 * variance ** 0.5                   # eta = 0 (prepare_extra_step_kwargs(generator, 0.0), :330)
            c = N.dh_ddim_coeffs(float(guidance_scale), float(beta_t ** 0.5), float(alpha_t ** 0.5), float(alpha_prev ** 0.5),
                                 float((1 - alpha_prev - std_dev_t ** 2) ** 0.5), 1 if divide_by_reciprocal else 0)
            self._coeffs[key] = c
        return c


def _flat_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise N.NativeLibraryError(f"{name} must live on a CUDA device (got {t.device}); there is no CPU path")
    t = t.detach()
    if t.dtype is not torch.float32 or not t.is_contiguous():
        t = t.to(torch.float32).contiguous()
    return t


def latent_step(latents: torch.Tensor, grad: torch.Tensor, step_size: float = 0.1, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``latents - grad * step_size`` (guided_stable_diffuser.py:434) in one launch; ``out`` may be ``latents`` (in place)."""
    lat, g = _flat_f32(latents, "latents"), _flat_f32(grad, "grad")
    if lat.shape != g.shape:
        raise ValueError(f"latents {tuple(lat.shape)} and grad {tuple(g.shape)} differ in shape")
    if out is None:
        out = torch.empty_like(lat)
    elif out.shape != lat.shape or out.dtype is not torch.float32 or not out.is_contiguous() or out.device != lat.device:
        raise ValueError("out must be a contiguous fp32 tensor of the latents' shape on the same device")
    N.check(N.load().dh_latent_step(lat.data_ptr(), g.data_ptr(), float(step_size), out.data_ptr(), lat.numel(),
                                    N.stream_handle(lat.device)), "dh_latent_step")
    return out


def cfg_ddim_step(noise_uncond: torch.Tensor, noise_text: Optional[torch.Tensor], sample: torch.Tensor, coeffs: N.dh_ddim_coeffs,
                  out: Optional[torch.Tensor] = None, eps_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Classifier-free-guidance combine + DDIM update in one launch (guided_stable_diffuser.py:470-474):
    ``eps = uncond + s (text - uncond)``; ``x0 = (sample - sqrt(1 - a_t) eps) / sqrt(a_t)``; returns
    ``sqrt(a_prev) x0 + sqrt(1 - a_prev) eps``.  ``noise_text=None``: plain DDIM update of ``noise_uncond``."""
    x = _flat_f32(sample, "sample")
    u = _flat_f32(noise_uncond, "noise_uncond")
    t = _flat_f32(noise_text, "noise_text") if noise_text is not None else None
    if u.numel() != x.numel() or (t is not None and t.numel() != x.numel()):
        raise ValueError("the noise predictions and the sample differ in size")
    if out is None:
        out = torch.empty_like(x)
    for name, o in (("out", out), ("eps_out", eps_out)):
        if o is not None and (o.numel() != x.numel() or o.dtype is not torch.float32 or not o.is_contiguous() or o.device != x.device):
            raise ValueError(f"{name} must be a contiguous fp32 tensor of the sample's size on the same device")
    N.check(N.load().dh_cfg_ddim_step(u.data_ptr(), t.data_ptr() if t is not None else None, x.data_ptr(), C.byref(coeffs), out.data_ptr(),
                                      eps_out.data_ptr() if eps_out is not None else None, x.numel(), N.stream_handle(x.device)),
            "dh_cfg_ddim_step")
    return out


def guided_denoise(latents: torch.Tensor, timesteps: Sequence, unet: Callable, scheduler_step: Optional[Callable],
                   activations_orig: List[torch.Tensor], processed_correspondences,
                   fg_weight: float = 1.5, bg_weight: float = 1.25, num_optsteps: int = 3, guidance_max_step: int = 38,
                   guidance_schedule_type: str = "constant", bg_loss_type: str = "global_avg", fg_patch_size: int = 1,
                   bg_patch_size: int = 1, step_size: float = 0.1, scale_model_input: Optional[Callable] = None,
                   cfg_noise: Optional[Callable] = None, skip_zero_weight_layers: bool = False,
                   on_step: Optional[Callable] = None, ddim: Optional[DDIMSchedule] = None, cfg_pair: Optional[Callable] = None,
                   guidance_scale: float = 7.5) -> torch.Tensor:
    """latents (1,4,h,w).  ``unet(latents_in, t) -> (noise_pred, [act0, act1, act2])`` with activations (1,C,h,w) that are
    differentiable w.r.t. ``latents_in``; ``scheduler_step(noise_pred, t, latents) -> latents``;
    ``cfg_noise(latents, t, t_idx) -> noise_pred`` runs the classifier-free-guidance forward (defaults to ``unet``).

    With ``ddim`` (a ``DDIMSchedule`` whose timesteps are set) and ``cfg_pair(latents, t, t_idx) -> (noise_uncond, noise_text)``
    the guidance combine and the scheduler update are ONE launch (``cfg_ddim_step``) and ``scheduler_step`` / ``cfg_noise`` are not
    called; ``cfg_pair`` may return ``(noise, None)`` for a plain DDIM update.

    guided_stable_diffuser.py:415-434: loss = sum_l fgw[l] * L_fg,l + bgw[l] * L_bg,l; latents -= 0.1 * dloss/dlatents.
    """
    return _denoise(False, latents, timesteps, unet, scheduler_step, activations_orig, processed_correspondences, fg_weight,
                    bg_weight, num_optsteps, guidance_max_step, guidance_schedule_type, bg_loss_type, fg_patch_size, bg_patch_size,
                    step_size, scale_model_input, cfg_noise, skip_zero_weight_layers, on_step, ddim, cfg_pair, guidance_scale)


def guided_denoise_batch(latents: torch.Tensor, timesteps: Sequence, unet: Callable, scheduler_step: Optional[Callable],
                         activations_orig, processed_correspondences: Sequence,
                         fg_weight: float = 1.5, bg_weight: float = 1.25, num_optsteps: int = 3, guidance_max_step: int = 38,
                         guidance_schedule_type: str = "constant", bg_loss_type: str = "global_avg", fg_patch_size: int = 1,
                         bg_patch_size: int = 1, step_size: float = 0.1, scale_model_input: Optional[Callable] = None,
                         cfg_noise: Optional[Callable] = None, skip_zero_weight_layers: bool = False,
                         on_step: Optional[Callable] = None, ddim: Optional[DDIMSchedule] = None, cfg_pair: Optional[Callable] = None,
                         guidance_scale: float = 7.5) -> torch.Tensor:
    """``guided_denoise`` for B edits at once: latents (B,4,h,w), ``processed_correspondences`` holds B dicts, and the callables
    see all B edits (``unet`` returns activations (B,C,h,w)).  ``activations_orig`` is one identity (three (T,C,h,w) stacks)
    shared by every edit, or a list of B identities.  Per guided iteration: one U-Net forward at batch B, one batched loss
    launch (``guidance_loss_and_grad_batch``), one backward and one ``latent_step``; per timestep one ``cfg_ddim_step`` (all
    edits share the timestep, so one set of coefficients serves them).

    The backward runs on the sum of the per-edit losses.  Its gradient w.r.t. edit e's latents is edit e's own gradient as long
    as the U-Net mixes no samples of the batch, which Stable Diffusion's U-Net (GroupNorm, per-sample attention) does not; a
    model with batch statistics (BatchNorm in training mode) would break that.  'local_avg' with different foreground and
    background patch sizes (the autograd path of ``guided_denoise``) is not implemented here."""
    if bg_loss_type == 'local_avg' and bg_patch_size != fg_patch_size:
        raise NotImplementedError("guided_denoise_batch: 'local_avg' with different fg / bg patch sizes is not implemented")
    if latents.dim() != 4 or latents.shape[0] != len(processed_correspondences):
        raise ValueError(f"latents must be (B,4,h,w) with B = {len(processed_correspondences)} edits, got {tuple(latents.shape)}")
    return _denoise(True, latents, timesteps, unet, scheduler_step, activations_orig, list(processed_correspondences), fg_weight,
                    bg_weight, num_optsteps, guidance_max_step, guidance_schedule_type, bg_loss_type, fg_patch_size, bg_patch_size,
                    step_size, scale_model_input, cfg_noise, skip_zero_weight_layers, on_step, ddim, cfg_pair, guidance_scale)


def _denoise(batch, latents, timesteps, unet, scheduler_step, activations_orig, processed_correspondences, fg_weight, bg_weight,
             num_optsteps, guidance_max_step, guidance_schedule_type, bg_loss_type, fg_patch_size, bg_patch_size, step_size,
             scale_model_input, cfg_noise, skip_zero_weight_layers, on_step, ddim, cfg_pair, guidance_scale):
    """The loop of ``guided_denoise`` (batch=False: one edit) and ``guided_denoise_batch`` (batch=True: B edits)."""
    schedule = make_guidance_weight_schedule(fg_weight, bg_weight, guidance_max_step, guidance_schedule_type)
    fused_update = ddim is not None and cfg_pair is not None
    if not fused_update and scheduler_step is None:
        raise ValueError("either scheduler_step or (ddim, cfg_pair) is required")
    if fused_update:           # the timestep values index the coefficient table on the host: one read-back for the whole loop
        t_host = [int(v) for v in (timesteps.tolist() if isinstance(timesteps, (torch.Tensor, np.ndarray)) else timesteps)]
    # batch mode: one identity shared by every edit, or one identity per edit (the loss kernel reads each edit's per-step slice in
    # place; edits of one scene may share an identity)
    per_edit_orig = batch and not isinstance(activations_orig[0], torch.Tensor)
    ident = activations_orig[0] if per_edit_orig else activations_orig
    for t_idx, t in enumerate(timesteps):
        iteration = 0
        while iteration < num_optsteps and t_idx < guidance_max_step:
            with torch.enable_grad():
                lat = latents.detach().requires_grad_(True)
                model_in = scale_model_input(lat, t) if scale_model_input is not None else lat
                _, activations = unet(model_in, t)
                fgw, bgw = schedule(t_idx, iteration)
                acts = list(activations) if batch else [a[0] for a in activations]
                if per_edit_orig:
                    origs = [[ao[l][t_idx] for ao in activations_orig] for l in range(len(acts))]
                else:
                    origs = [a[t_idx] for a in activations_orig]
                activations_size = (ident[2][t_idx].shape[-2], ident[2][t_idx].shape[-1])
                if skip_zero_weight_layers:       # a zero-weight layer contributes exactly 0 (the reference still evaluates it)
                    keep = [i for i in range(len(acts)) if fgw[i] != 0.0 or bgw[i] != 0.0]
                    acts, origs = [acts[i] for i in keep], [origs[i] for i in keep]
                    fgw, bgw = [fgw[i] for i in keep], [bgw[i] for i in keep]
                grad = None
                if acts and (bg_loss_type != 'local_avg' or bg_patch_size == fg_patch_size):
                    # value and d(loss)/d(activations) from one fused launch; the U-Net's backward then carries them to the latents
                    # (the chain rule of autograd.grad(loss, latents), guided_stable_diffuser.py:430-434)
                    loss_and_grad = guidance_loss_and_grad_batch if batch else guidance_loss_and_grad
                    _, _, act_grads = loss_and_grad(acts, origs, processed_correspondences, fgw, bgw, bg_loss_type=bg_loss_type,
                                                    activations_size=activations_size, patch_size=fg_patch_size)
                    grad = torch.autograd.grad(acts, [lat], grad_outputs=act_grads)[0]
                elif acts:
                    loss, _ = guidance_loss(acts, origs, processed_correspondences, fgw, bgw, bg_loss_type=bg_loss_type,
                                            activations_size=activations_size, patch_size=fg_patch_size,
                                            bg_patch_size=bg_patch_size)
                    grad = torch.autograd.grad(loss, [lat])[0]
                if grad is not None:
                    latents = latent_step(lat, grad, step_size)         # latents - grad * 0.1 (:434), one launch
            iteration += 1
        if on_step is not None:
            on_step('opt', latents)
        with torch.no_grad():
            if fused_update:
                noise_uncond, noise_text = cfg_pair(latents, t, t_idx)
                latents = cfg_ddim_step(noise_uncond, noise_text, latents, ddim.coefficients(t_host[t_idx], guidance_scale)).view(latents.shape)
            else:
                noise_pred = cfg_noise(latents, t, t_idx) if cfg_noise is not None else unet(latents, t)[0]
                latents = scheduler_step(noise_pred, t, latents)
            if on_step is not None:
                on_step('post-opt', latents)
    return latents
