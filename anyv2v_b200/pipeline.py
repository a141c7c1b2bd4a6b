"""I2VGen-XL sampling loops, B200-native: ``invert`` and ``sample_with_pnp``.

Drop-in for the two hot loops of the reference's ``I2VGenXLPipeline`` (i2vgen-xl/pipelines/pipeline_i2vgen_xl.py):
  invert            :1197-1439 (loop :1385-1433)
  sample_with_pnp   :892-1195  (loop :1131-1179)
with the same keyword surface for everything that reaches the loops.  Differences, none of which changes a result:
  * no host sync inside the loop: timesteps are Python ints (the reference calls ``t.item()`` at :1143 and runs
    ``t in tensor`` membership kernels inside every hook), inverted latents stay in HBM (anyv2v_b200.latent_store)
    instead of ``torch.save``/``torch.load`` per step (:1134, :1424-1428);
  * conditioning that does not depend on t (fps embedding, 145-token context, image-latent stem) is computed once
    per clip (``unet.precompute_conditioning``) instead of once per step;
  * CFG + scheduler step is one fused kernel (``scheduler.step(..., model_output_cond=...)``);
  * on steps where no injection fires, the source branch — whose prediction the reference discards at :1160 — is
    not run at all (every norm is per-sample, so the edit branches do not depend on it).
CLIP / VAE encoders are outside the hot path and the metric (SURVEY 8d, 8f rank 4): the loops take pre-encoded
tensors (``prompt_embeds``, ``image_embeddings``, ``image_latents`` ...) or — with ``encoders=`` (anyv2v_b200.encoders)
and ``vae=`` attached — the reference's raw inputs (prompt strings, PIL first frames), encoded once per clip.
"""
from __future__ import annotations

import logging
import os
from types import SimpleNamespace
from typing import Callable, Optional

import torch

from .latent_store import LatentStore
from .pnp_utils import _fires, register_time

logger = logging.getLogger(__name__)


def frame_position_latents(first_frame_latent: torch.Tensor, num_frames: int) -> torch.Tensor:
    """prepare_image_latents (pipeline :532-562) minus the VAE: [b,4,h,w] -> [b,4,F,h,w], frame k>=1 = k/(F-1)."""
    x = first_frame_latent.unsqueeze(2)
    if num_frames == 1:
        return x
    scale = torch.arange(1, num_frames, device=x.device, dtype=torch.float32) / (num_frames - 1)
    mask = torch.ones_like(x).expand(-1, -1, num_frames - 1, -1, -1) * scale.view(1, 1, -1, 1, 1).to(x.dtype)
    return torch.cat([x, mask], dim=2)


class _GraphedIteration:
    """One loop iteration captured as a CUDA graph (streams + graphs instead of a tracing compiler).

    The iteration body reads only static device buffers (latents, source latent, timestep, scheduler coefficients) so
    the same graph is replayed for every timestep with the same hook-flag combination.  The first use runs eagerly
    (allocates workspaces / packed weights, builds nothing under capture), the second captures, later ones replay."""

    def __init__(self, body, on_cuda: bool = True, pool=None):
        self.body = body      # () -> None, operating on static buffers
        self.graph = None
        self.calls = 0
        self.on_cuda = bool(on_cuda)   # where the body's tensors live (NOT whether the box has a GPU)
        self.pool = pool               # shared memory pool of the per-hook-flag graphs of one loop

    def run(self):
        self.calls += 1
        if self.calls == 1 or not self.on_cuda:
            self.body()
            return
        if self.graph is None:
            g = torch.cuda.CUDAGraph()
            # thread_local: the latent-store writer thread may call cudaEventSynchronize while this thread captures
            with torch.cuda.graph(g, pool=self.pool, capture_error_mode="thread_local"):
                self.body()
            self.graph = g
        self.graph.replay()


def tensor2vid(video: torch.Tensor, output_type: str = "np"):
    """pipeline_i2vgen_xl.py:79-97 with diffusers' `VaeImageProcessor.postprocess` (do_normalize=True) inlined:
    video [b, 3, f, H, W] in [-1, 1] -> "pt": [b, f, 3, H, W] in [0, 1]; "np": float32 [b, f, H, W, 3]; "pil": list (per
    batch entry) of lists of PIL images."""
    if output_type not in ("np", "pt", "pil"):
        raise ValueError(f"{output_type} does not exist. Please choose one of ['np', 'pt', 'pil]")
    outputs = []
    for batch_vid in video.permute(0, 2, 1, 3, 4):             # [f, 3, H, W] per batch entry
        img = (batch_vid / 2 + 0.5).clamp(0, 1)
        if output_type == "pt":
            outputs.append(img)
            continue
        arr = img.detach().cpu().permute(0, 2, 3, 1).float().numpy()
        if output_type == "np":
            outputs.append(arr)
        else:
            from PIL import Image
            outputs.append([Image.fromarray(a) for a in (arr * 255).round().astype("uint8")])
    if output_type == "np":
        import numpy as np
        return np.stack(outputs)
    if output_type == "pt":
        return torch.stack(outputs)
    return outputs


class I2VGenXLPipeline:
    #: replay loop iterations as CUDA graphs (set False to run every kernel launch eagerly)
    use_cuda_graphs = os.environ.get("AV2V_CUDA_GRAPHS", "1") != "0"

    def __init__(self, unet, scheduler=None, encoders: Optional[SimpleNamespace] = None, vae=None):
        self.unet = unet
        self.scheduler = scheduler
        self.vae = vae  # optional anyv2v_b200.vae.AutoencoderKL (or any module with diffusers' encode/decode protocol)
        self.encoders = encoders  # optional: .encode_prompt(str)->[1,77,D], .encode_image(img)->[1,1,D], .encode_vae(img)->[1,4,h,w]
        self.latent_store: Optional[LatentStore] = None
        self._guidance_scale = 1.0

    # -- small diffusers-pipeline surface the runners touch ---------------------------------------------------------
    @property
    def device(self):
        return next(self.unet.parameters()).device

    _execution_device = device

    @property
    def do_classifier_free_guidance(self):
        return self._guidance_scale > 1

    def to(self, device):
        self.unet.to(device)
        return self

    # -- the steps either side of the loops (SURVEY 8f row 4) ------------------------------------------------------
    def decode_latents(self, latents, decode_chunk_size=None):
        """pipeline_i2vgen_xl.py:443-463."""
        if self.vae is None:
            raise ValueError("decode_latents needs a VAE: construct the pipeline with `vae=` (anyv2v_b200.vae.AutoencoderKL)")
        from . import vae as vae_mod
        return vae_mod.decode_latents(self.vae, latents, decode_chunk_size)

    def encode_vae_video(self, video, device=None, height: Optional[int] = None, width: Optional[int] = None, generator=None):
        """pipeline_i2vgen_xl.py:565-592: ``video`` is the reference's list of PIL frames (each center-cropped-wide to
        (width, height) and mapped to [-1, 1], :578-580) or an already pre-processed tensor [f, 3, H, W] in [-1, 1];
        -> video latents [1, 4, f, H/8, W/8].  All frames go through the VAE in one batch."""
        if self.vae is None:
            raise ValueError("encode_vae_video needs a VAE: construct the pipeline with `vae=`")
        from . import image_io
        from . import vae as vae_mod
        if not torch.is_tensor(video):
            if height is None or width is None:
                width, height = video[0].size
            video = image_io.preprocess(image_io.center_crop_wide(list(video), (width, height)))
        p0 = next(self.vae.parameters())
        return vae_mod.encode_vae_video(self.vae, video.to(device=p0.device, dtype=p0.dtype), generator)

    # -- once-per-clip conditioning from raw inputs (pipeline :1318-1352 / :1014-1094) ----------------------------
    def encode_prompt(self, prompt):
        """pipeline :219-394 for this path (one prompt string, no LoRA, no clip_skip) -> [1, 77, D]."""
        if self.encoders is None:
            raise ValueError("a prompt STRING was given but the pipeline has no `encoders` (anyv2v_b200.encoders.ClipEncoders): "
                             "attach them or pass `prompt_embeds`")
        return self.encoders.encode_prompt(prompt).to(self.device)

    def encode_first_frame(self, image, height: int, width: int, num_frames: int, generator=None):
        """The image half of the conditioning: CLIP image embedding of the square crop (:1318-1322, `_encode_image`
        :395-412) and the VAE latent of the (width, height) crop with the frame-position planes appended
        (`prepare_image_latents` :532-562) -> (image_embeddings [1, 1, D], image_latents [1, 4, F, h, w])."""
        if self.encoders is None or self.vae is None:
            raise ValueError("a first-frame IMAGE was given but the pipeline lacks `encoders` and/or `vae`: attach them or pass "
                             "`image_embeddings` / `image_latents`")
        from . import image_io
        emb = self.encoders.encode_image(image, width).to(self.device)
        x = image_io.preprocess(image_io.center_crop_wide(image, (width, height))).to(device=self.device, dtype=next(self.vae.parameters()).dtype)
        lat = self.vae.encode(x).latent_dist.sample(generator) * self.vae.config.scaling_factor
        return emb, frame_position_latents(lat.to(emb.dtype), num_frames)

    def _size_of(self, image, height, width):
        if (height is None or width is None) and image is not None and hasattr(image, "size"):
            width, height = image.size
        return height, width

    def register_modules(self, **kwargs):
        for k, v in kwargs.items():
            setattr(self, k, v)

    def check_inputs(self, prompt_embeds, image_latents, image_embeddings, latents):
        # mirrors the ValueError convention of pipeline :483-530 for the tensors this path takes
        for name, t in (("prompt_embeds", prompt_embeds), ("image_latents", image_latents),
                        ("image_embeddings", image_embeddings), ("latents", latents)):
            if t is None:
                raise ValueError(f"`{name}` is required: pass it pre-encoded, or give the raw prompt / image to a pipeline built "
                                 f"with `encoders=` (anyv2v_b200.encoders.ClipEncoders) and `vae=`.")
        if latents.dim() != 5 or latents.shape[1] != self.unet.config["in_channels"]:
            raise ValueError(f"`latents` must be [b, {self.unet.config['in_channels']}, f, h, w], got {tuple(latents.shape)}")
        if image_latents.shape[2:] != latents.shape[2:]:
            raise ValueError("`image_latents` and `latents` must agree in (frames, h, w)")
        # every down block halves the latent and its up block doubles it back: odd sizes on the way down cannot be restored
        f = 2 ** (len(self.unet.config["block_out_channels"]) - 1)
        h, w = latents.shape[3], latents.shape[4]
        if h % f or w % f:
            raise ValueError(f"latent size {h} x {w} is not divisible by {f}: frame sides must be multiples of {8 * f} px "
                             f"(64 px for I2VGen-XL, e.g. 1280 x 704), got {8 * w} x {8 * h} px")

    def _any_hook_fires(self, t) -> bool:
        mod = self.unet.up_blocks[1].resnets[1]
        if _fires(t, getattr(mod, "_injection_set", None)):
            return True
        for res in (1, 2, 3):
            up = self.unet.up_blocks[res]
            for blk in range(3):
                for proc in (up.attentions[blk].transformer_blocks[0].attn1.processor,
                             up.temp_attentions[blk].transformer_blocks[0].attn1.processor):
                    if _fires(t, getattr(proc, "_injection_set", None)):
                        return True
        return False

    # -- phase 1 --------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def invert(self, prompt=None, image=None, height=None, width=None, target_fps: int = 16, num_frames: int = 16,
               num_inference_steps: int = 50, guidance_scale: float = 1.0, negative_prompt=None, eta: float = 0.0,
               latents: Optional[torch.Tensor] = None, prompt_embeds=None, negative_prompt_embeds=None,
               image_embeddings=None, image_latents=None, output_dir: Optional[str] = None, return_dict: bool = False,
               write_files: bool = True, callback: Optional[Callable] = None, max_steps: Optional[int] = None,
               host_resident: bool = False, **_ignored):
        """DDIM inversion x_0 -> x_T (pipeline :1385-1433).  Returns [b, steps, c, f, h, w] in DESCENDING-t order like
        the reference (:1436); every x_t is kept in ``self.latent_store`` (and written as ddim_latents_{t}.pt)."""
        if prompt_embeds is None and prompt is not None:
            prompt_embeds = self.encode_prompt(prompt)
        if guidance_scale > 1 and negative_prompt_embeds is None:
            negative_prompt_embeds = self.encode_prompt(negative_prompt if negative_prompt is not None else "")  # :348-352
        if image is not None and (image_embeddings is None or image_latents is None):
            height, width = self._size_of(image, height, width)
            emb, lat = self.encode_first_frame(image, height, width, num_frames)
            image_embeddings = emb if image_embeddings is None else image_embeddings
            image_latents = lat if image_latents is None else image_latents
        st = self.prepare_invert(latents, prompt_embeds, image_latents, image_embeddings, target_fps,
                                 num_inference_steps, guidance_scale, output_dir, write_files, host_resident,
                                 negative_prompt_embeds=negative_prompt_embeds)
        n = len(st.timesteps) if max_steps is None else min(max_steps, len(st.timesteps))
        inverted = []
        for i in range(n):
            self.invert_step(st, i)
            inverted.append(st.store.get(st.timesteps[i], device=st.latents.device))
            if callback is not None:
                callback(i, st.timesteps[i], st.latents)
        st.store.flush()
        stacked = torch.stack(list(reversed(inverted)), 1)
        return SimpleNamespace(frames=stacked) if return_dict else stacked

    def prepare_invert(self, latents, prompt_embeds, image_latents, image_embeddings, target_fps, num_inference_steps,
                       guidance_scale=1.0, output_dir=None, write_files=True, host_resident=False,
                       negative_prompt_embeds=None):
        """Everything of ``invert`` that happens once per clip (pipeline :1316-1382).  With ``guidance_scale > 1`` the
        step runs the UNet on [uncond, cond] (:1387-1388: negative prompt, zero image embedding :420-422, same image
        latents :559-560) and combines them (:1407-1410) inside the fused inverse-DDIM kernel."""
        self._guidance_scale = guidance_scale
        self.check_inputs(prompt_embeds, image_latents, image_embeddings, latents)
        cfg = self.do_classifier_free_guidance
        if cfg and negative_prompt_embeds is None:
            raise ValueError("`negative_prompt_embeds` (or a `negative_prompt` string + encoders) is required when guidance_scale > 1")
        dev = self.device
        latents = latents.to(dev)
        if cfg and latents.shape[0] != 1:
            raise ValueError("inversion with guidance handles one clip per call (the reference's batch is always 1, :571)")
        d = lambda x: x.to(dev)
        if cfg:
            fps = torch.tensor([target_fps] * 2, device=dev)
            cond = self.unet.precompute_conditioning(fps, torch.cat([d(image_latents)] * 2),
                                                     torch.cat([torch.zeros_like(d(image_embeddings)), d(image_embeddings)]),
                                                     torch.cat([d(negative_prompt_embeds), d(prompt_embeds)]))
        else:
            fps = torch.tensor([target_fps], device=dev).repeat(latents.shape[0])
            cond = self.unet.precompute_conditioning(fps, d(image_latents), d(image_embeddings), d(prompt_embeds))
        self.scheduler.set_timesteps(num_inference_steps, device=dev)
        ts = self.scheduler.timesteps.tolist()
        store = LatentStore(output_dir, write_files=write_files, host_resident=host_resident)
        self.latent_store = store
        st = SimpleNamespace(latents=latents.contiguous().clone(), cond=cond, timesteps=ts, store=store, scheduler=self.scheduler)
        st.t_table = torch.tensor(ts, device=dev, dtype=torch.int64)
        st.coef_table = self.scheduler.coefficient_table(ts, guidance_scale if cfg else 1.0, dev)
        st.g_t = torch.zeros(1, device=dev, dtype=torch.int64)
        st.g_coef = torch.zeros(5, device=dev, dtype=torch.float32)

        if cfg:
            def body():
                v = self.unet(torch.cat([st.latents, st.latents]), st.g_t, cond=st.cond)[0]
                st.scheduler.step(v[0:1], None, st.latents, model_output_cond=v[1:2], out=st.latents, coef_dev=st.g_coef)
        else:
            def body():
                v = self.unet(st.latents, st.g_t, cond=st.cond)[0]
                st.scheduler.step(v, None, st.latents, out=st.latents, coef_dev=st.g_coef)  # in place: x_t -> x_{t+1}

        st.iteration = _GraphedIteration(body, on_cuda=st.latents.is_cuda)
        return st

    def invert_step(self, st, i: int):
        """One iteration of the inversion loop (pipeline :1385-1433): UNet (B = 1) -> inverse DDIM step -> keep x_t."""
        t = st.timesteps[i]
        st.g_t.copy_(st.t_table[i:i + 1])
        st.g_coef.copy_(st.coef_table[i])
        if self.use_cuda_graphs:
            st.iteration.run()
        else:
            st.iteration.body()
        st.store.put(t, st.latents)
        return st.latents

    # -- phase 2 --------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def sample_with_pnp(self, prompt=None, image=None, height=None, width=None, target_fps: int = 16,
                        num_frames: int = 16, num_inference_steps: int = 50, guidance_scale: float = 9.0,
                        negative_prompt=None, eta: float = 0.0, generator=None, latents: Optional[torch.Tensor] = None,
                        prompt_embeds=None, negative_prompt_embeds=None, output_type: str = "latent",
                        return_dict: bool = True, ddim_init_latents_t_idx: int = 1,
                        ddim_inv_latents_path: Optional[str] = None, ddim_inv_prompt=None, ddim_inv_1st_frame=None,
                        ddim_inv_prompt_embeds=None, image_embeddings=None, image_latents=None,
                        ddim_inv_image_embeddings=None, ddim_inv_image_latents=None,
                        latent_store: Optional[LatentStore] = None, skip_dead_source_branch: bool = True,
                        callback: Optional[Callable] = None, max_steps: Optional[int] = None,
                        decode_chunk_size: Optional[int] = None, **_ignored):
        """PnP edit loop (pipeline :1131-1179) over the branches [source, uncond, cond]; `output_type` "latent" returns
        the latents, "pt" / "np" / "pil" decode them with the attached VAE (:1180-1194)."""
        # raw inputs (the reference's only interface, :1014-1094) are encoded once per clip when encoders / VAE are attached
        if prompt_embeds is None and prompt is not None:
            prompt_embeds = self.encode_prompt(prompt)
        if negative_prompt_embeds is None and (negative_prompt is not None or prompt is not None):
            negative_prompt_embeds = self.encode_prompt(negative_prompt if negative_prompt is not None else "")
        if ddim_inv_prompt_embeds is None and ddim_inv_prompt is not None:
            ddim_inv_prompt_embeds = self.encode_prompt(ddim_inv_prompt)
        if image is not None and (image_embeddings is None or image_latents is None):
            height, width = self._size_of(image, height, width)
            emb, lat = self.encode_first_frame(image, height, width, num_frames, generator)
            image_embeddings = emb if image_embeddings is None else image_embeddings
            image_latents = lat if image_latents is None else image_latents
        if ddim_inv_1st_frame is not None and (ddim_inv_image_embeddings is None or ddim_inv_image_latents is None):
            height, width = self._size_of(ddim_inv_1st_frame, height, width)
            emb, lat = self.encode_first_frame(ddim_inv_1st_frame, height, width, num_frames, generator)
            ddim_inv_image_embeddings = emb if ddim_inv_image_embeddings is None else ddim_inv_image_embeddings
            ddim_inv_image_latents = lat if ddim_inv_image_latents is None else ddim_inv_image_latents
        st = self.prepare_edit(latents, prompt_embeds, negative_prompt_embeds, ddim_inv_prompt_embeds, image_embeddings,
                               image_latents, ddim_inv_image_embeddings, ddim_inv_image_latents, target_fps,
                               num_inference_steps, guidance_scale, ddim_init_latents_t_idx, ddim_inv_latents_path,
                               latent_store, skip_dead_source_branch)
        n = len(st.timesteps) if max_steps is None else min(max_steps, len(st.timesteps))
        for i in range(n):
            self.edit_step(st, i)
            if callback is not None:
                callback(i, st.timesteps[i], st.latents)
        if output_type == "latent":
            return SimpleNamespace(frames=st.latents) if return_dict else (st.latents,)
        video = tensor2vid(self.decode_latents(st.latents, decode_chunk_size=decode_chunk_size), output_type)
        return SimpleNamespace(frames=video) if return_dict else (video,)

    def prepare_edit(self, latents, prompt_embeds, negative_prompt_embeds, ddim_inv_prompt_embeds, image_embeddings,
                     image_latents, ddim_inv_image_embeddings, ddim_inv_image_latents, target_fps, num_inference_steps,
                     guidance_scale, ddim_init_latents_t_idx=0, ddim_inv_latents_path=None, latent_store=None,
                     skip_dead_source_branch=True):
        """Everything of ``sample_with_pnp`` that happens once per clip (pipeline :1014-1128)."""
        self._guidance_scale = guidance_scale
        if not self.do_classifier_free_guidance:
            raise NotImplementedError("the PnP edit path runs with classifier-free guidance (cfg 9.0)")
        self.check_inputs(prompt_embeds, image_latents, image_embeddings, latents)
        for name, t in (("negative_prompt_embeds", negative_prompt_embeds), ("ddim_inv_prompt_embeds", ddim_inv_prompt_embeds),
                        ("ddim_inv_image_embeddings", ddim_inv_image_embeddings), ("ddim_inv_image_latents", ddim_inv_image_latents)):
            if t is None:
                raise ValueError(f"`{name}` is required (pre-encoded)")
        dev = self.device
        # explicit arguments win: a store left on the pipeline by an earlier invert() of ANOTHER clip must not shadow the
        # path the caller names (the reference only knows `ddim_inv_latents_path`, pipeline :1134)
        if latent_store is not None:
            store = latent_store
        elif ddim_inv_latents_path is not None:
            mine = self.latent_store
            same = (mine is not None and mine.output_dir is not None
                    and os.path.abspath(mine.output_dir) == os.path.abspath(ddim_inv_latents_path))
            store = mine if same else LatentStore(ddim_inv_latents_path, write_files=False)
        elif self.latent_store is not None:
            store = self.latent_store
        else:
            raise ValueError("need `latent_store` or `ddim_inv_latents_path`")
        d = lambda x: x.to(dev)
        # [source, uncond, cond] stacks (:1043-1046, :1093-1101); uncond image embedding is zeros (:438)
        prompts3 = torch.cat([d(ddim_inv_prompt_embeds), d(negative_prompt_embeds), d(prompt_embeds)])
        img_emb3 = torch.cat([d(ddim_inv_image_embeddings), torch.zeros_like(d(image_embeddings)), d(image_embeddings)])
        img_lat3 = torch.cat([d(ddim_inv_image_latents), d(image_latents), d(image_latents)])
        fps3 = torch.tensor([target_fps] * 3, device=dev)
        cond3 = self.unet.precompute_conditioning(fps3, img_lat3, img_emb3, prompts3)
        self.scheduler.set_timesteps(num_inference_steps, device=dev)
        ts = self.scheduler.timesteps.tolist()[ddim_init_latents_t_idx:]
        logger.info("Sampling starts from latents_at_t=%s", ts[0] if ts else None)
        fires = [self._any_hook_fires(t) for t in ts]
        cond2 = None
        if skip_dead_source_branch and not all(fires):
            cond2 = {k: v[v.shape[0] // 3:].contiguous() for k, v in cond3.items()}  # every entry is branch-major
        st = SimpleNamespace(latents=d(latents).contiguous().clone(), cond3=cond3, cond2=cond2, timesteps=ts, store=store,
                             fires=fires, guidance=guidance_scale, skip=skip_dead_source_branch, scheduler=self.scheduler)
        st.t_table = torch.tensor(ts, device=dev, dtype=torch.int64)
        st.coef_table = self.scheduler.coefficient_table(ts, guidance_scale, dev)
        st.g_t = torch.zeros(1, device=dev, dtype=torch.int64)
        st.g_coef = torch.zeros(5, device=dev, dtype=torch.float32)
        st.g_src = torch.zeros_like(st.latents)
        st.iterations = {}  # hook-flag combination -> _GraphedIteration
        st.graph_pool = torch.cuda.graph_pool_handle() if st.latents.is_cuda else None  # one activation pool for all of them
        # uncond and cond are the same latents + image latents -> they share the UNet prefix up to the first cross-attention
        # (I2VGenXLUNet.forward, shared_edit_prefix); the source branch is dropped after the last injection site that fires in
        # the step (its prediction is discarded, pipeline :1160).  Both leave the result unchanged (measured +2.3 % / +0.9 % on
        # the bench schedule, profiles/r02_probe.txt; `skip_dead_source_branch=False` runs the reference's full batch instead)
        st.shared_prefix = bool(skip_dead_source_branch)
        st.prune_source = bool(skip_dead_source_branch)
        return st

    def _hook_flags(self, t):
        """Which of the three injections fire at t (decided on the host; baked into the captured graph)."""
        mod = self.unet.up_blocks[1].resnets[1]
        up = self.unet.up_blocks[3]
        spa = up.attentions[2].transformer_blocks[0].attn1.processor
        tmp = up.temp_attentions[2].transformer_blocks[0].attn1.processor
        return (_fires(t, getattr(mod, "_injection_set", None)), _fires(t, getattr(spa, "_injection_set", None)),
                _fires(t, getattr(tmp, "_injection_set", None)))

    @staticmethod
    def _prune_site(flags):
        """(conv, spatial, temporal) flags of a step -> the last site at which the source branch is still read
        (UNet order inside a layer: resnet -> temp_conv -> spatial transformer -> temporal transformer; the hooks sit on
        up_blocks[1].resnets[1] and on attentions / temp_attentions of up_blocks[1..3], pnp_utils.py:130,235,340)."""
        conv, spatial, temporal = flags
        if temporal:
            return (3, 2, "temporal")
        if spatial:
            return (3, 2, "spatial")
        if conv:
            return (1, 1, "resnet")
        return None

    def edit_step(self, st, i: int):
        """One iteration of the PnP edit loop (pipeline :1131-1179)."""
        t = st.timesteps[i]
        register_time(self, t)
        dead_source = st.skip and not st.fires[i]
        key = (dead_source,) + self._hook_flags(t)
        it = st.iterations.get(key)
        if it is None:
            if dead_source:
                def body():
                    v = self.unet(torch.cat([st.latents, st.latents]), st.g_t, cond=st.cond2,
                                  shared_edit_prefix=st.shared_prefix)[0]
                    st.scheduler.step(v[0:1], None, st.latents, model_output_cond=v[1:2], out=st.latents, coef_dev=st.g_coef)
            else:
                site = self._prune_site(key[1:]) if st.prune_source else None
                lo = 0 if site is not None else 1  # the pruned forward returns [uncond, cond] only

                def body():
                    v = self.unet(torch.cat([st.g_src, st.latents, st.latents]), st.g_t, cond=st.cond3,
                                  shared_edit_prefix=st.shared_prefix, prune_source_after=site)[0]
                    st.scheduler.step(v[lo:lo + 1], None, st.latents, model_output_cond=v[lo + 1:lo + 2], out=st.latents,
                                      coef_dev=st.g_coef)
            it = st.iterations[key] = _GraphedIteration(body, on_cuda=st.latents.is_cuda, pool=st.graph_pool)
        st.g_t.copy_(st.t_table[i:i + 1])
        st.g_coef.copy_(st.coef_table[i])
        if not dead_source:
            st.g_src.copy_(st.store.get(t, device=st.latents.device), non_blocking=True)
        if self.use_cuda_graphs:
            it.run()
        else:
            it.body()
        return st.latents
