"""``DiffusionHandles`` facade with the reference's method names and signatures (diffusion_handles.py:13-166).

The geometry half of ``transform_foreground`` (:143-149) runs on the sm_100a kernels of this package.  The
diffusion half (U-Net, VAE, text encoder, scheduler, null-text inversion) is stock PyTorch/diffusers code that this
build deliberately does not re-implement (north star): it is injected as ``diffuser`` / ``inverter`` objects that
expose the reference's ``initial_inference`` / ``guided_inference`` / ``invert`` methods.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch

from .depth_transform import (_as_scene, _scene_planes, normalize_depth, transform_depth, transform_depth_mesh_scenes, transform_depth_pc_objects,
                              transform_depth_pc_scenes)
from .guided_stable_diffuser import GuidedStableDiffuser

DEFAULT_CONF = SimpleNamespace(   # diffhandles/config/default.yaml
    guided_diffuser=SimpleNamespace(bg_weight=1.25, fg_weight=1.5, fg_patch_size=1, bg_patch_size=1, use_depth=True,
                                    save_denoising_steps=False, bg_loss_type='global_avg', num_timesteps=50, num_optsteps=3,
                                    guidance_max_step=38, guidance_schedule_type='constant', bg_erosion=0, seed=2773),
    depth_transform_mode='pc')


class DiffusionHandles:
    def __init__(self, conf=None, diffuser=None, inverter=None):
        self.conf = DEFAULT_CONF if conf is None else conf
        self.diffuser = GuidedStableDiffuser(conf=self.conf.guided_diffuser) if diffuser is None else diffuser
        self.inverter = inverter
        self.device = torch.device('cpu')

    def to(self, device: torch.device = None):
        self.diffuser.to(device=device)
        if self.inverter is not None:
            self.inverter.to(device=device)
        self.device = device
        return self

    def _need(self, obj, method):
        if obj is None or not hasattr(obj, method):
            raise NotImplementedError(
                f"{method} needs the stock-PyTorch diffusion model (U-Net / VAE / scheduler), which is outside this build; "
                "pass a diffuser / inverter object that implements it")
        return getattr(obj, method)

    def invert_input_image(self, img: torch.Tensor, depth: torch.Tensor, prompt: str):
        disparity = normalize_depth(1.0 / depth)
        _, init_noise, null_text_emb = self._need(self.inverter, "invert")(
            target_img=img, depth=disparity, prompt=prompt, num_inner_steps=5, verbose=True)
        return null_text_emb, init_noise

    def generate_input_image(self, depth: torch.Tensor, prompt: str, null_text_emb: torch.Tensor = None,
                             init_noise: torch.Tensor = None):
        disparity = normalize_depth(1.0 / depth)
        with torch.no_grad():
            activations, latent_image, null_text_emb, init_noise = self._need(self.diffuser, "initial_inference")(
                init_latents=init_noise, depth=disparity, uncond_embeddings=null_text_emb, prompt=prompt)
        return null_text_emb, init_noise, activations, latent_image

    def set_foreground(self, depth: torch.Tensor, fg_mask: torch.Tensor, bg_depth: torch.Tensor) -> torch.Tensor:
        """diffusion_handles.py:88-110: background depth = input depth with the (15 px dilated) foreground hole filled by
        a Poisson problem driven by the Laplacian of ``bg_depth``.  Entirely on the device: the dilation is one pass of the
        bit-packed morphology kernel with the 31 x 31 diamond that 15 iterations of SciPy's cross element amount to.  Runs as
        ``set_foreground_scenes`` with one scene.  For a multi-object edit (``transform_foreground_objects``) pass the union of
        the object masks: the background is filled under every object at once."""
        H, W = depth.shape[-2:]
        return self.set_foreground_scenes(_as_scene(depth, H, W), _as_scene(fg_mask, H, W), _as_scene(bg_depth, H, W))

    def set_foreground_scenes(self, depths: torch.Tensor, fg_masks: torch.Tensor, bg_depths: torch.Tensor) -> torch.Tensor:
        """``set_foreground`` for S scenes of one size ((S,1,H,W) tensors or sequences of S (1,1,H,W) tensors): one dilation launch
        and one Poisson launch for all of them (the S systems are independent).  Returns (S,1,H,W); entry s equals
        ``set_foreground`` of scene s bit for bit."""
        from . import _native as N
        from .depth_transform import _pack_mask, _poisson_device
        depths, fg_masks, bg_depths = (_scene_planes(x, n) for x, n in ((depths, "depths"), (fg_masks, "fg_masks"), (bg_depths, "bg_depths")))
        S, H, W = depths.shape[0], depths.shape[-2], depths.shape[-1]
        for name, t in (("fg_masks", fg_masks), ("bg_depths", bg_depths)):
            if tuple(t.shape) != (S, 1, H, W):
                raise ValueError(f"{name} must be {(S, 1, H, W)} like depths, got {tuple(t.shape)}")
        lib = N.load()
        dev = depths.device
        d = depths.reshape(S, H, W).to(torch.float32).contiguous()
        b = bg_depths.reshape(S, H, W).to(device=dev, dtype=torch.float32).contiguous()
        bits = _pack_mask((fg_masks.reshape(S, H, W).to(dev) != 0).to(torch.float32).contiguous())
        r = 15
        rows = N.u32_array([((1 << (2 * (r - abs(i - r)) + 1)) - 1) << abs(i - r) for i in range(2 * r + 1)])
        dil = torch.empty_like(bits)
        N.check(lib.dh_morph_pass(N.ptr(bits), N.ptr(dil), S, H, W, rows, 2 * r + 1, 2 * r + 1, 1, N.stream_handle(dev)), "dh_morph_pass")
        # (the reference's set_foreground is synchronous CPU code: the convergence check's small read-back costs nothing extra)
        return _poisson_device(d, dil, lap_source=b, check=True, what="set_foreground")[:, None]

    def edit_geometry(self, depth: torch.Tensor, fg_mask: torch.Tensor, bg_depth: torch.Tensor, rot_angle: float = None,
                      rot_axis: torch.Tensor = None, translation: torch.Tensor = None, use_input_depth_normalization=False):
        """The geometry half of an edit on the sm_100a kernels: edited disparity (1,1,H,W) and correspondences (N,4) int64."""
        with torch.no_grad():
            return transform_depth(depth=depth, bg_depth=bg_depth, fg_mask=fg_mask,
                                   intrinsics=self.diffuser.get_depth_intrinsics(device=depth.device), rot_angle=rot_angle,
                                   rot_axis=rot_axis, translation=translation,
                                   use_input_depth_normalization=use_input_depth_normalization,
                                   depth_transform_mode=self.conf.depth_transform_mode)

    def transform_foreground(self, depth: torch.Tensor, prompt: str, fg_mask: torch.Tensor, bg_depth: torch.Tensor,
                             null_text_emb: torch.Tensor, init_noise: torch.Tensor, activations: list,
                             rot_angle: float = None, rot_axis: torch.Tensor = None, translation: torch.Tensor = None,
                             fg_weight: float = None, bg_weight: float = None, use_input_depth_normalization=False):
        """diffusion_handles.py:110-166: geometry on this package's kernels, then the injected diffuser's guided denoising.
        Returns (edited_img, edited_disparity) plus the saved denoising steps when the configuration asks for them."""
        guided = self._need(self.diffuser, "guided_inference")
        disparity, correspondences = self.edit_geometry(depth, fg_mask, bg_depth, rot_angle, rot_axis, translation,
                                                        use_input_depth_normalization)
        keep_steps = bool(self.conf.guided_diffuser.save_denoising_steps)
        with torch.no_grad():
            out = guided(latents=init_noise, depth=disparity, uncond_embeddings=null_text_emb, prompt=prompt,
                         activations_orig=activations, correspondences=correspondences, fg_weight=fg_weight,
                         bg_weight=bg_weight, save_denoising_steps=keep_steps)
        if keep_steps:
            image, steps = out
            return image, disparity, steps
        return out, disparity

    def edit_geometry_batch(self, depth: torch.Tensor, fg_mask: torch.Tensor, bg_depth: torch.Tensor, rot_angles, rot_axes,
                            translations, use_input_depth_normalization=False):
        """B transforms of one scene: ``edit_geometry_scenes`` with one scene.  Edited disparities (B,1,H,W) and a list of B
        correspondence lists, each equal bit for bit to ``edit_geometry`` with that transform."""
        H, W = depth.shape[-2:]
        return self.edit_geometry_scenes([_as_scene(depth, H, W)], [_as_scene(fg_mask, H, W)], [_as_scene(bg_depth, H, W)], [0] * len(rot_angles),
                                         rot_angles, rot_axes, translations, use_input_depth_normalization)

    def edit_geometry_scenes(self, depths, fg_masks, bg_depths, scene_index, rot_angles, rot_axes, translations,
                             use_input_depth_normalization=False):
        """B edits over S scenes of one size (``depths`` / ``fg_masks`` / ``bg_depths`` (S,1,H,W) or sequences of S (1,1,H,W)
        tensors; edit b transforms scene ``scene_index[b]``).  In 'pc' mode the edits are ONE ``EditEngine`` batch
        (``transform_depth_pc_scenes``), in 'mesh' mode ONE ``dh_edit_mesh_scenes`` call (``transform_depth_mesh_scenes``).
        Returns (disparities (B,1,H,W), [correspondences (n_b,4) int64 CPU] * B), entry b equal bit for bit to ``edit_geometry``
        of its scene with its transform."""
        scenes = {"pc": transform_depth_pc_scenes, "mesh": transform_depth_mesh_scenes}.get(self.conf.depth_transform_mode)
        if scenes is None:
            raise ValueError(f"Unknown depth transform mode '{self.conf.depth_transform_mode}'.")
        dev = (depths if isinstance(depths, torch.Tensor) else depths[0]).device
        with torch.no_grad():
            return scenes(depths, bg_depths, fg_masks, self.diffuser.get_depth_intrinsics(device=dev), scene_index, rot_angles, rot_axes,
                          translations, use_input_depth_normalization)

    def transform_foreground_batch(self, depth: torch.Tensor, prompt: str, fg_mask: torch.Tensor, bg_depth: torch.Tensor,
                                   null_text_emb: torch.Tensor, init_noise: torch.Tensor, activations: list, rot_angles, rot_axes,
                                   translations, fg_weight: float = None, bg_weight: float = None, use_input_depth_normalization=False):
        """``transform_foreground`` for B transforms of one scene: ``transform_foreground_scenes`` with one scene, whose prompt,
        ``init_noise`` and identity ``activations`` every edit shares.  Returns (edited images (B,...), edited disparities
        (B,1,H,W)).  Saving the denoising steps is not supported in batch mode."""
        H, W = depth.shape[-2:]
        return self.transform_foreground_scenes([_as_scene(depth, H, W)], [prompt], [_as_scene(fg_mask, H, W)], [_as_scene(bg_depth, H, W)],
                                                [null_text_emb], [init_noise], [activations], [0] * len(rot_angles), rot_angles, rot_axes,
                                                translations, fg_weight, bg_weight, use_input_depth_normalization)

    def transform_foreground_scenes(self, depths, prompts, fg_masks, bg_depths, null_text_embs, init_noises, identities, scene_index,
                                    rot_angles, rot_axes, translations, fg_weight: float = None, bg_weight: float = None,
                                    use_input_depth_normalization=False):
        """``transform_foreground`` for B edits over S scenes: the geometry of all edits in one batch (``edit_geometry_scenes``),
        then ONE ``guided_inference_batch`` in which edit b takes the prompt, null-text sequence, initial noise and identity of
        its scene ``scene_index[b]`` (``prompts``, ``null_text_embs``, ``init_noises``, ``identities``: one entry per scene; the
        identities are referenced, never copied).  When every edit is of one scene, that scene's values are passed as shared
        ones.  Returns (edited images (B,...), edited disparities (B,1,H,W)).  Saving the denoising steps is not supported in
        batch mode."""
        guided = self._need(self.diffuser, "guided_inference_batch")
        if self.conf.guided_diffuser.save_denoising_steps:
            raise NotImplementedError("transform_foreground_batch does not save the denoising steps; use transform_foreground per edit")
        S = len(depths)
        for name, v in (("prompts", prompts), ("null_text_embs", null_text_embs), ("init_noises", init_noises), ("identities", identities)):
            if len(v) != S:
                raise ValueError(f"{name} must have one entry per scene ({S}), got {len(v)}")
        disparities, correspondences = self.edit_geometry_scenes(depths, fg_masks, bg_depths, scene_index, rot_angles, rot_axes,
                                                                 translations, use_input_depth_normalization)
        index = [int(i) for i in scene_index]
        if len(set(index)) == 1:
            s = index[0]
            prompt, uncond, latents, acts = prompts[s], null_text_embs[s], init_noises[s], identities[s]
        else:
            prompt = [prompts[s] for s in index]
            if not all(isinstance(p, str) for p in prompt):
                prompt = torch.cat([prompts[s] for s in index])              # per-edit embedding rows (B,L,D)
            uncond = [null_text_embs[s] for s in index]
            latents = torch.cat([init_noises[s] for s in index])
            acts = [identities[s] for s in index]
        with torch.no_grad():
            images = guided(latents=latents, depth=disparities, uncond_embeddings=uncond, prompt=prompt, activations_orig=acts,
                            correspondences=correspondences, fg_weight=fg_weight, bg_weight=bg_weight)
        return images, disparities

    def edit_geometry_objects(self, depth: torch.Tensor, fg_masks, bg_depth: torch.Tensor, rot_angles, rot_axes, translations,
                              use_input_depth_normalization=False):
        """The geometry of one edit that moves K disjoint objects of the image, each by its own transform
        (``transform_depth_pc_objects``; ``fg_masks`` (K,1,H,W) or K (1,1,H,W) masks, ``rot_angles`` etc. of length K).  Returns
        (edited disparity (1,1,H,W), correspondences (N,4) int64).  'pc' mode only."""
        if self.conf.depth_transform_mode != "pc":
            raise NotImplementedError(f"multi-object edits run in 'pc' mode only, not '{self.conf.depth_transform_mode}'")
        with torch.no_grad():
            return transform_depth_pc_objects(depth, bg_depth, fg_masks, self.diffuser.get_depth_intrinsics(device=depth.device),
                                              rot_angles, rot_axes, translations, use_input_depth_normalization)

    def transform_foreground_objects(self, depth: torch.Tensor, prompt: str, fg_masks, bg_depth: torch.Tensor, null_text_emb: torch.Tensor,
                                     init_noise: torch.Tensor, activations: list, rot_angles, rot_axes, translations,
                                     fg_weight: float = None, bg_weight: float = None, use_input_depth_normalization=False):
        """``transform_foreground`` for K objects moved at once: the geometry of ``edit_geometry_objects``, then ONE guided
        denoising pass of the injected diffuser over the joint correspondences (the losses see one list, as for a single
        object).  ``bg_depth`` is ``set_foreground`` of the union of the masks.  Returns (edited_img, edited_disparity) plus the
        saved denoising steps when the configuration asks for them.  'pc' mode only."""
        guided = self._need(self.diffuser, "guided_inference")
        disparity, correspondences = self.edit_geometry_objects(depth, fg_masks, bg_depth, rot_angles, rot_axes, translations,
                                                                use_input_depth_normalization)
        keep_steps = bool(self.conf.guided_diffuser.save_denoising_steps)
        with torch.no_grad():
            out = guided(latents=init_noise, depth=disparity, uncond_embeddings=null_text_emb, prompt=prompt,
                         activations_orig=activations, correspondences=correspondences, fg_weight=fg_weight,
                         bg_weight=bg_weight, save_denoising_steps=keep_steps)
        if keep_steps:
            image, steps = out
            return image, disparity, steps
        return out, disparity
