"""SVITalkVideoPipeline — SVI with per-frame audio conditioning (reference diffsynth/pipelines/svi_video_talk.py).

Differences to SVIVideoPipeline, as in the reference: the DiT is an `enable_multitalk` WanModel whose blocks carry an
audio cross-attention (wan_video_dit.py:339-366); the clip's wav2vec window features [1, num_frames, 5, 12, 768] are split
into a first-frame window and per-latent-frame windows (`preprocess_audio`, :432-446), projected once per clip
(`WanDiTEngine.audio_state`) and fed to every forward; guidance is three-way (:448-466):

    v = v_uncond + s_text * (v_cond - v_drop_text) + s_audio * (v_drop_text - v_uncond)

with v_cond (prompt, audio), v_drop_text (negative prompt, audio), v_uncond (negative prompt, silent audio).
The window features come from `audio_path` (a WAV file) through the native wav2vec2 encoder
(utils/src/audio_analysis/wav2vec2.py, loaded lazily from `wav2vec_path`, default ./weights/chinese-wav2vec2-base/ as in the
reference), or are passed in directly as `audio_embed`.  The embedding of the whole file is kept on the device for the
next call with the same file (keyed by real path, size and mtime), so chained clips encode their audio once.
"""
import os

import torch
from PIL import Image
from tqdm import tqdm

from .svi_video import SVIVideoPipeline, TeaCache


def preprocess_audio(audio_embed, audio_window=5, vae_scale=4):
    """[1, 4n+1, w, 12, 768] window features -> (first frame [1,1,w,12,768], latter frames [1,n,w+vae_scale-1,12,768]):
    inside each group of `vae_scale` video frames the first keeps windows 0..mid, the last mid..w-1, the others their
    centre window (reference :432-446)."""
    first = audio_embed[:, :1]
    rest = audio_embed[:, 1:]
    b, n4, w, s, c = rest.shape
    if n4 % vae_scale:
        raise ValueError(f"audio features must cover 4n+1 frames, got {n4 + 1}")
    rest = rest.reshape(b, n4 // vae_scale, vae_scale, w, s, c)
    mid = audio_window // 2
    head = rest[:, :, :1, :mid + 1].reshape(b, n4 // vae_scale, -1, s, c)
    tail = rest[:, :, -1:, mid:].reshape(b, n4 // vae_scale, -1, s, c)
    centre = rest[:, :, 1:-1, mid:mid + 1].reshape(b, n4 // vae_scale, -1, s, c)
    return first, torch.cat([head, centre, tail], dim=2)


def model_fn_wan_talk_video(dit, x, timestep, context, clip_feature=None, y=None, tea_cache=None, add_condition=None,
                            audio_embed_tuple=None, use_unified_sequence_parallel=False, use_controlnet=False, **kwargs):
    """Drop-in for reference svi_video_talk.py:82-157: one forward of the enable_multitalk DiT, result in x.dtype.
    `audio_embed_tuple` may also be an AudioState (pre-projected audio)."""
    sp = None
    if use_unified_sequence_parallel:
        from ..distributed.sequence_parallel import get_sp_group
        sp = get_sp_group()
    eng = dit.engine(x.device if x.is_cuda else None)
    out = eng.forward(x, timestep, context, clip_feature, y, sp=sp, tea_cache=tea_cache, add_condition=add_condition,
                      audio=audio_embed_tuple)
    return out.to(x.dtype)


class SVITalkVideoPipeline(SVIVideoPipeline):
    def __init__(self, device="cuda", torch_dtype=torch.float16, tokenizer_path=None, wav2vec_path=None, is_test=False):
        super().__init__(device=device, torch_dtype=torch_dtype, tokenizer_path=tokenizer_path, is_test=is_test)
        self.wav2vec_path = wav2vec_path
        self.wav2vec_feature_extractor, self.audio_encoder = None, None
        self._audio_cache = None          # ((realpath, size, mtime_ns), [S, layers, 768] f32 on the device)

    @staticmethod
    def from_model_manager(model_manager, torch_dtype=None, device=None, use_usp=False, is_test=False, wav2vec_path=None):
        device = model_manager.device if device is None else device
        torch_dtype = model_manager.torch_dtype if torch_dtype is None else torch_dtype
        pipe = SVITalkVideoPipeline(device=device, torch_dtype=torch_dtype, wav2vec_path=wav2vec_path, is_test=is_test)
        pipe.fetch_models(model_manager)
        if use_usp:
            pipe.enable_usp()
        return pipe

    def load_audio_encoder(self):
        """custom_init (reference :26-30): feature extractor + encoder from `wav2vec_path`, on first use."""
        if self.audio_encoder is None:
            from utils.src.audio_analysis.wav2vec2 import Wav2Vec2FeatureExtractor, Wav2Vec2Model
            path = self.wav2vec_path if self.wav2vec_path is not None else "./weights/chinese-wav2vec2-base/"
            if not os.path.isdir(path):
                raise FileNotFoundError(f"wav2vec2 checkpoint directory not found: {os.path.abspath(path)} "
                                        f"(pass wav2vec_path=, or audio_embed= with precomputed window features)")
            self.wav2vec_feature_extractor = Wav2Vec2FeatureExtractor.from_pretrained(path, local_files_only=True)
            self.audio_encoder = Wav2Vec2Model.from_pretrained(path, local_files_only=True)
        return self.wav2vec_feature_extractor, self.audio_encoder

    def audio_embedding(self, audio_path):
        """[S, layers, 768] f32 on the device for the whole file; recomputed only when the file changes."""
        from utils.audio_process import audio_prepare_single, embedding_device
        st = os.stat(audio_path)
        key = (os.path.realpath(audio_path), st.st_size, st.st_mtime_ns)
        if self._audio_cache is None or self._audio_cache[0] != key:
            fe, enc = self.load_audio_encoder()
            self._audio_cache = None
            emb = embedding_device(audio_prepare_single(audio_path), fe, enc, device=self.device)
            self._audio_cache = (key, emb)
        return self._audio_cache[1]

    def get_audio_embedding(self, audio_path, num_frames, audio_start_idx=0):
        """reference :412-430: [1, num_frames, 5, layers, 768] window features of frames audio_start_idx .. + num_frames,
        window rows clamped to the audio; every rank of a use_usp group computes the same bits (no atomics on the path)."""
        from utils.audio_process import cut_windows
        return cut_windows(self.audio_embedding(audio_path), num_frames, audio_start_idx)

    def preprocess_audio(self, audio_embed, audio_window=5, vae_scale=4):
        first, latter = preprocess_audio(audio_embed, audio_window, vae_scale)
        return first.to(self.device).to(torch.bfloat16), latter.to(self.device).to(torch.bfloat16)

    def denoise_latents_talk(self, latents, context_posi, context_nega, clip_feature, y, audio_embed_tuple, audio_embed_tuple_null,
                             cfg_scale, progress_bar_cmd=lambda x: x, tea_cache_posi=None, tea_cache_nega=None, condition=None):
        """reference _sample_with_multitalk :448-466 (three forwards per step unless both scales are 1)."""
        eng = self.dit.engine(self.device)
        # three-way guidance: the forwards of one step run one after the other on every rank, each split over the token axis
        # of the rank's sequence-parallel group (with two CFG groups both groups compute the same step)
        sp = self.sp_group()
        sp = sp if sp is not None and sp.sp_size > 1 else None
        lat = latents if latents.dtype == torch.float32 and latents.is_contiguous() else latents.to(torch.float32).contiguous()
        if y is not None:
            y = y.to(device=self.device, dtype=torch.float32).contiguous()
        cp = eng.context_state(context_posi, clip_feature)
        cn = eng.context_state(context_nega, clip_feature)
        audio = eng.audio_state(audio_embed_tuple)
        silent = eng.audio_state(audio_embed_tuple_null)
        st, sa = float(cfg_scale["text"]), float(cfg_scale["audio"])
        v_c, v_u, v_d = torch.empty_like(lat), torch.empty_like(lat), torch.empty_like(lat)
        sig, ts = self.scheduler.sigmas, self.scheduler.timesteps
        n = len(ts)
        for i in progress_bar_cmd(range(n)):
            t = float(ts[i])
            eng.forward(lat, t, cp, y=y, sp=sp, out=v_c, tea_cache=tea_cache_posi, add_condition=condition, audio=audio)
            if st != 1.0 or sa != 1.0:
                # the reference hands the SAME nega TeaCache to both of these calls (:457-458); kept
                eng.forward(lat, t, cn, y=y, sp=sp, out=v_u, tea_cache=tea_cache_nega, audio=silent)
                eng.forward(lat, t, cn, y=y, sp=sp, out=v_d, tea_cache=tea_cache_nega, add_condition=condition, audio=audio)
                # v = v_u + st (v_c - v_d) + sa (v_d - v_u) = st v_c + (sa - st) v_d + (1 - sa) v_u
                eng.k.axpby(v_c, st, v_d, sa - st, v_c)
                eng.k.axpby(v_c, 1.0, v_u, 1.0 - sa, v_c)
            nxt = float(sig[i + 1]) if i + 1 < n else 0.0
            eng.k.axpby(lat, 1.0, v_c, nxt - float(sig[i]), lat)        # Euler: x += v (sigma_next - sigma), flow_match.py:63
        return lat

    @torch.no_grad()
    def __call__(self, prompt, negative_prompt="", input_image=None, input_video=None, denoising_strength=1.0, seed=None,
                 rand_device="cpu", height=480, width=832, num_frames=81, cfg_scale=5.0, num_inference_steps=50,
                 sigma_shift=5.0, tiled=True, tile_size=(30, 52), tile_stride=(15, 26), tea_cache_l1_thresh=None,
                 tea_cache_model_id="", progress_bar_cmd=tqdm, random_ref_frame=None, audio_path=None, use_controlnet=False,
                 audio_start_idx=0, args=None, audio_embed=None):
        height, width = self.check_resize_height_width(height, width)
        if num_frames % 4 != 1:
            num_frames = (num_frames + 2) // 4 * 4 + 1
            print(f"Only `num_frames % 4 != 1` is acceptable. We round it up to {num_frames}.")
        if not isinstance(cfg_scale, dict) or "audio" not in cfg_scale:
            raise ValueError("SVI-Talk takes cfg_scale=dict(text=..., audio=...) (reference svi_video_talk.py:456-462)")
        tiler_kwargs = {"tiled": tiled, "tile_size": tile_size, "tile_stride": tile_stride}
        self.scheduler.set_timesteps(num_inference_steps, denoising_strength=denoising_strength, shift=sigma_shift)
        noise = self.generate_noise((1, 16, (num_frames - 1) // 4 + 1, height // 8, width // 8), seed=seed,
                                    device=rand_device, dtype=torch.float32)
        latents = noise.to(dtype=self.torch_dtype, device=self.device).to(torch.float32)
        if input_video is not None:
            vid = torch.stack(self.preprocess_images(input_video), dim=2).to(dtype=torch.float32, device=self.device)
            latents = self.scheduler.add_noise(self.encode_video(vid, **tiler_kwargs).to(torch.float32), latents,
                                               timestep=self.scheduler.timesteps[0])
        pos = self.encode_prompt(prompt, positive=True)
        neg = self.encode_prompt(negative_prompt, positive=False)
        image_emb = {}
        if input_image is not None and self.image_encoder is not None:
            ref_img = Image.fromarray(random_ref_frame.clone().cpu().numpy())
            if not isinstance(input_image, list):
                input_image = [input_image]
            image_emb = self.encode_images_adaptive(input_image, ref_img, num_frames, height, width, use_first_aug=False,
                                                    ref_pad_cfg=args.ref_pad_cfg, ref_pad_num=args.ref_pad_num)
        if audio_embed is None:
            audio_embed = self.get_audio_embedding(audio_path, num_frames, audio_start_idx=audio_start_idx)
        if tuple(audio_embed.shape[:2]) != (1, num_frames):
            raise ValueError(f"audio_embed must be [1, {num_frames}, 5, 12, 768], got {tuple(audio_embed.shape)}")
        audio_tuple = self.preprocess_audio(audio_embed)
        # reference :550: `torch.zeros_like(audio_embed)[-1:]` keeps the batch entry, i.e. an all-zero feature clip
        audio_null = self.preprocess_audio(torch.zeros_like(audio_embed)[-1:])
        mk = lambda: (TeaCache(num_inference_steps, rel_l1_thresh=tea_cache_l1_thresh, model_id=tea_cache_model_id)
                      if tea_cache_l1_thresh is not None else None)
        bar = (lambda r: progress_bar_cmd(r)) if progress_bar_cmd is not None else (lambda r: r)
        latents = self.denoise_latents_talk(latents, pos["context"], neg["context"], image_emb.get("clip_feature"),
                                            image_emb.get("y"), audio_tuple, audio_null, cfg_scale, bar, mk(), mk())
        frames = self.decode_video(latents, **tiler_kwargs)
        return self.tensor2video(frames[0])
