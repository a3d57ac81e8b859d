"""TEST / BENCH INFRASTRUCTURE — stand-in for the text-to-video path of the reference's ``GenerationSession``
(release_server.py:344-736) on boxes where the reference checkout (and its FastAPI / omegaconf dependencies)
does not exist: ``bench.py``, ``smoke()`` and the ``-m gpu`` tests drive the server's per-block sequence
through it.  In a real deployment the reference's OWN ``GenerationSession`` runs unmodified on the drop-in
classes; ``tests/golden/reference_callers_small.npz`` records exactly that (unmodified release_server.py, bit-equal
with this stand-in block by block when recorded), ``tests/test_reference_callers_cpu.py`` checks this stand-in
against the record, and ``tests/golden/server_loop_small.npz`` holds the same loop executed by the reference
modules alone.

Per block (release_server.py:636-736):
    recompute_kv_cache  -> block >= 1: re-initialise the cache, one DiT pass at t=0 over the
                           kv_cache_num_frames clean context frames under the block-causal mask
    N denoise steps     -> DiT pass, flow->x0, re-noise with the session RNG (bf16 randn)
    VAE decode          -> pixels [1, 12, 3, H, W] fp32 in [-1, 1] (block 0: 9 frames decoded, the first 3 skipped)
Webcam / v2v / prompt interpolation / start-frame are caller features outside the hot path.
Once the context window slides, the reference re-encodes the oldest cached PIXEL frame into the first
context latent (release_server.py:571-576; at 832x480 its bicubic resize to 480x832 is the identity): done
with ``models.vae_encoder``; with ``keep_first_frame=True`` the first latent frame is kept (:566-570).
"""
from __future__ import annotations

from collections import deque
from dataclasses import dataclass
from typing import Optional

import torch

from realtime_video_b200.wan_wrapper import FlowMatchScheduler


@dataclass
class GenerateParams:
    """Fields of release_server.py:315-341 that the text-to-video path reads."""
    prompt: str = ""
    width: int = 832
    height: int = 480
    seed: int = 42
    kv_cache_num_frames: int = 3
    num_blocks: int = 9
    num_denoising_steps: int = 4
    timestep_shift: float = 5.0
    strength: float = 1.0
    keep_first_frame: bool = False
    context_noise: float = 0.0


def get_denoising_schedule(timesteps: torch.Tensor, denoising_strength: float, steps: int = 4):
    """v2v.py:133-136."""
    lst = torch.linspace(denoising_strength * 1000, 0, steps, dtype=torch.float32,
                         device=timesteps.device).to(torch.long)
    return timesteps[1000 - lst]


class Models:
    """release_server.py:100-109."""

    def __init__(self, text_encoder, transformer, pipeline, vae_encoder, vae_decoder):
        self.text_encoder, self.transformer, self.pipeline = text_encoder, transformer, pipeline
        self.vae_encoder, self.vae_decoder = vae_encoder, vae_decoder


class GenerationSession:
    @torch.inference_mode()          # like the reference (release_server.py:347): the caches it resets are inference tensors
    def __init__(self, params: GenerateParams, models: Models, prompt_embeds: Optional[torch.Tensor] = None,
                 device=None, decode: bool = True):
        self.params, self.models, self.decode = params, models, decode
        # one stream on several GPUs (sequence-parallel or layer-pipelined): rank 0 decodes for everybody
        self.decode_enabled = decode or self._multi_gpu_mode(models) is not None
        self.gpu = torch.device(device if device is not None else "cuda")
        self.width, self.height = params.width // 8 * 8, params.height // 8 * 8
        self.latent_width, self.latent_height = self.width // 8, self.height // 8
        self.num_frame_per_block = 3
        self.num_blocks = params.num_blocks
        self.block_idx = 0
        self.current_start_frame = 0
        self.frame_context_cache = deque(maxlen=1 + (params.kv_cache_num_frames - 1) * 4)
        self.decode_vae_cache = [None] * 55
        self.rnd = torch.Generator(self.gpu).manual_seed(params.seed)
        shape = [1, self.num_blocks * self.num_frame_per_block, 16, self.latent_height, self.latent_width]
        self.all_latents = torch.zeros(shape, device=self.gpu, dtype=torch.bfloat16)
        self.noise = torch.randn(shape, device=self.gpu, dtype=torch.bfloat16, generator=self.rnd)
        self.conditional_dict = None
        if prompt_embeds is not None:
            self.conditional_dict = {"prompt_embeds": prompt_embeds.to(self.gpu, torch.bfloat16).contiguous()}
        self.init_models()
        self.denoising_step_list = get_denoising_schedule(self.zero_padded_timesteps, params.strength,
                                                          steps=params.num_denoising_steps)
        self.last_pred = None

    @staticmethod
    def _multi_gpu_mode(models):
        m = models.pipeline.generator.model
        sp, pp = getattr(m, "sp", None), getattr(m, "pp", None)
        return sp if sp is not None else pp

    # release_server.py:542-560
    def init_models(self):
        p = self.models.pipeline
        p.frame_seq_length = (self.latent_height // 2) * (self.latent_width // 2)
        for block in p.generator.model.blocks:
            block.self_attn.local_attn_size = -1
        p.local_attn_size = self.params.kv_cache_num_frames + p.num_frame_per_block
        p._initialize_kv_cache(batch_size=1, dtype=torch.bfloat16, device=self.gpu)
        p._initialize_crossattn_cache(batch_size=1, dtype=torch.bfloat16, device=self.gpu)
        p.generator.model.block_mask = None
        p.scheduler = FlowMatchScheduler(shift=self.params.timestep_shift, sigma_min=0.0, extra_one_step=True)
        p.scheduler.set_timesteps(1000, training=True)
        st = p.scheduler.timesteps
        self.zero_padded_timesteps = torch.cat((st.cpu(), torch.tensor([0], dtype=torch.float32))).to(self.gpu)

    # release_server.py:563-576
    def get_clean_context_frames(self):
        kvn = self.params.kv_cache_num_frames
        nfpb = self.models.pipeline.num_frame_per_block
        ctx = self.all_latents[:, :self.current_start_frame]
        keep = self.params.keep_first_frame or self.models.vae_encoder is None or not self.decode_enabled
        if keep or (self.block_idx - 1) * nfpb < kvn:
            if kvn == 1:
                return ctx[:, :1]
            return torch.cat((ctx[:, :1], ctx[:, 1:][:, -kvn + 1:]), dim=1)
        # window has slid: first context latent = re-encoded oldest cached pixel frame
        ctx = ctx[:, 1:][:, -kvn + 1:]
        first = None
        if self.decode:
            frame = self.frame_context_cache[0][0].half()                 # [1, 3, H, W]
            z = frame.transpose(0, 1).unsqueeze(0)                        # [1, 3, 1, H, W] (v2v.py:138-158)
            mu, _ = self.models.vae_encoder(z, [None] * 55, stream=False)
            first = mu.squeeze(0).to(torch.float16).transpose(0, 1)[None].to(self.all_latents)   # [1,1,16,h,w]
        par = self._multi_gpu_mode(self.models)
        if par is not None:                                               # one stream on several GPUs
            import torch.distributed as dist
            if first is None:
                first = torch.empty_like(ctx[:, :1])
            first = first.contiguous()
            src = 0 if par.group is None else dist.get_global_rank(par.group, 0)
            dist.broadcast(first, src=src, group=par.group)
        return torch.cat((first, ctx), dim=1)

    # release_server.py:588-633
    def recompute_kv_cache(self):
        p = self.models.pipeline
        if self.block_idx == 0:
            p._initialize_kv_cache(batch_size=1, dtype=torch.bfloat16, device=self.gpu)
            return self.current_start_frame
        for block in p.generator.model.blocks:
            block.self_attn.num_frame_per_block = p.num_frame_per_block
        kvn = self.params.kv_cache_num_frames
        model_input_start_frame = min(self.current_start_frame, kvn)
        ctx = self.get_clean_context_frames()
        p._initialize_kv_cache(batch_size=1, dtype=ctx.dtype, device=ctx.device)
        model = p.generator.model
        model.block_mask = model._prepare_blockwise_causal_attn_mask(
            device=str(ctx.device), num_frames=ctx.shape[1], frame_seqlen=p.frame_seq_length,
            num_frame_per_block=p.num_frame_per_block, local_attn_size=-1)
        ts = torch.zeros([1, ctx.shape[1]], device=ctx.device, dtype=torch.int64)
        try:
            self.models.transformer(noisy_image_or_video=ctx, conditional_dict=self.conditional_dict,
                                    timestep=ts, kv_cache=p.kv_cache1, crossattn_cache=p.crossattn_cache,
                                    current_start=model_input_start_frame * p.frame_seq_length)
        finally:
            model.block_mask = None
        return model_input_start_frame

    # release_server.py:636-736
    @torch.inference_mode()
    def generate_block(self):
        idx = self.block_idx
        if idx >= self.num_blocks:
            return None
        p = self.models.pipeline
        if self.conditional_dict is None:
            cd = self.models.text_encoder(text_prompts=[self.params.prompt])
            self.conditional_dict = {k: v.to(dtype=torch.bfloat16).contiguous() for k, v in cd.items()}
        start = self.recompute_kv_cache()
        nf = p.num_frame_per_block
        noisy_input = self.noise[:, self.current_start_frame:self.current_start_frame + nf]
        steps = self.denoising_step_list
        denoised_pred = None
        for index, current_timestep in enumerate(steps):
            timestep = torch.ones([1, nf], device=self.gpu, dtype=torch.int64) * current_timestep
            _, denoised_pred = self.models.transformer(
                noisy_image_or_video=noisy_input, conditional_dict=self.conditional_dict, timestep=timestep,
                kv_cache=p.kv_cache1, crossattn_cache=p.crossattn_cache,
                current_start=start * p.frame_seq_length)
            if index < len(steps) - 1:
                next_timestep = steps[index + 1]
                flat = denoised_pred.flatten(0, 1)
                noisy_input = p.scheduler.add_noise(
                    flat, torch.randn(*flat.shape, generator=self.rnd, device=flat.device, dtype=torch.bfloat16),
                    next_timestep * torch.ones([nf], device=self.gpu, dtype=torch.long)
                ).unflatten(0, denoised_pred.shape[:2])
        self.all_latents[:, self.current_start_frame:self.current_start_frame + nf] = denoised_pred
        self.last_pred = denoised_pred
        pixels = None
        if self.decode and self.models.vae_decoder is not None:
            pixels, self.decode_vae_cache = self.models.vae_decoder(denoised_pred.half(), *self.decode_vae_cache)
            self.frame_context_cache.extend(pixels.split(1, dim=1))
            if idx == 0:
                pixels = pixels[:, 3:]          # release_server.py:722-723
        self.current_start_frame += nf
        self.block_idx += 1
        return pixels if pixels is not None else denoised_pred
