"""Audio preparation of SVI-Talk (reference utils/audio_process.py) without librosa, pyloudnorm or transformers.

- `audio_prepare_single` reads a WAV file (scipy.io.wavfile, soundfile's sample conventions), mixes it to mono by the mean
  of its channels, resamples it to 16 kHz if needed and normalises its loudness to -23 LUFS, as the reference does with
  librosa.load + pyloudnorm (:67-75).  The resampler is scipy.signal.resample_poly (Kaiser-windowed polyphase FIR), not
  librosa's soxr_hq, so audio at another rate than 16 kHz is not bit-equal to the reference's; 16 kHz WAV input is.
  Video containers and compressed formats raise: the reference shells out to ffmpeg for those (:44-65); convert with
  `ffmpeg -i in.mp4 -vn -ac 1 -ar 16000 -acodec pcm_s16le out.wav` first.
- `loudness_norm` implements ITU-R BS.1770-4 integrated loudness (K-weighting, 400 ms blocks with 75 % overlap, -70 LUFS
  absolute and -10 LU relative gating) with the reference's passthrough when |loudness| > 100 (:10-16).  The K-weighting
  biquads are designed for the sample rate with the published formulas that reproduce the standard's 48 kHz
  coefficients; pyloudnorm's design differs in the last digits, which moves the gain by far less than the bf16 rounding
  of the embedding once the feature extractor's mean/variance normalisation has run (tests show this at +-1 dB).
- `get_embedding` (:18-41) runs the native encoder and returns [S, layers, 768] fp32 on the CPU, S = int(len / sr * 25).
- `cut_audio_embedding` (:79-108) is the training-side window cut.
"""
import os

import numpy as np
import torch

_VIDEO = (".mp4", ".mov", ".avi", ".mkv", ".webm")


def read_wav(path):
    """(float32 [n] mono, rate): int16 / 32768, 24- and 32-bit int / 2^31 (scipy returns 24-bit samples in the top bytes
    of an int32), uint8 (x - 128) / 128, float as stored; channels averaged."""
    from scipy.io import wavfile
    rate, data = wavfile.read(path)
    if data.dtype == np.int16:
        x = data.astype(np.float32) / 32768.0
    elif data.dtype == np.int32:
        x = (data.astype(np.float64) / 2147483648.0).astype(np.float32)
    elif data.dtype == np.uint8:
        x = (data.astype(np.float32) - 128.0) / 128.0
    elif data.dtype in (np.float32, np.float64):
        x = data.astype(np.float32)
    else:
        raise ValueError(f"{path}: unsupported WAV sample format {data.dtype}")
    if x.ndim == 2:
        x = x.mean(axis=1, dtype=np.float32)
    return x, int(rate)


def load_audio(path, sr=16000):
    """librosa.load(path, sr=sr) for WAV files: mono float32 at `sr` (resample_poly when the file's rate differs)."""
    ext = os.path.splitext(path)[1].lower()
    if ext != ".wav":
        raise ValueError(f"{path}: only WAV input is supported; the reference decodes {ext or 'this'} files with ffmpeg — "
                         f"convert first, e.g. `ffmpeg -i {os.path.basename(path)} -vn -ac 1 -ar {sr} -acodec pcm_s16le out.wav`")
    x, rate = read_wav(path)
    if rate != sr:
        from math import gcd
        from scipy.signal import resample_poly
        g = gcd(rate, sr)
        x = resample_poly(x.astype(np.float64), sr // g, rate // g).astype(np.float32)
    return x


def _k_weighting(rate):
    """BS.1770 pre-filter (high shelf) and RLB high-pass as two biquads (b, a) for `rate`."""
    f0, G, Q = 1681.974450955533, 3.999843853973347, 0.7071752369554196
    K = np.tan(np.pi * f0 / rate)
    Vh = 10.0 ** (G / 20.0)
    Vb = Vh ** 0.4996667741545416
    a0 = 1.0 + K / Q + K * K
    shelf = (np.array([(Vh + Vb * K / Q + K * K) / a0, 2.0 * (K * K - Vh) / a0, (Vh - Vb * K / Q + K * K) / a0]),
             np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0]))
    f0, Q = 38.13547087602444, 0.5003270373238773
    K = np.tan(np.pi * f0 / rate)
    a0 = 1.0 + K / Q + K * K
    hp = (np.array([1.0, -2.0, 1.0]), np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0]))
    return shelf, hp


def integrated_loudness(x, rate=16000):
    """ITU-R BS.1770-4 integrated loudness in LUFS of a mono (or [n, channels], channel weights 1) signal; -inf when every
    block is gated out (e.g. digital silence)."""
    from scipy.signal import lfilter
    x = np.asarray(x, dtype=np.float64)
    if x.ndim == 1:
        x = x[:, None]
    block, step = int(round(0.4 * rate)), int(round(0.1 * rate))
    if x.shape[0] < block:
        raise ValueError(f"audio must be at least 400 ms long for a loudness measurement, got {x.shape[0] / rate:.3f} s")
    for b, a in _k_weighting(rate):
        x = lfilter(b, a, x, axis=0)
    n_blocks = (x.shape[0] - block) // step + 1
    csum = np.concatenate([np.zeros((1, x.shape[1])), np.cumsum(x * x, axis=0)])
    starts = np.arange(n_blocks) * step
    z = (csum[starts + block] - csum[starts]) / block                 # [blocks, channels] mean squares
    zs = z.sum(axis=1)
    with np.errstate(divide="ignore"):
        lj = -0.691 + 10.0 * np.log10(zs)
    keep = lj > -70.0
    if not keep.any():
        return float("-inf")
    rel = -0.691 + 10.0 * np.log10(zs[keep].mean()) - 10.0
    keep &= lj > rel
    return float(-0.691 + 10.0 * np.log10(zs[keep].mean()))


def loudness_norm(audio_array, sr=16000, lufs=-23):
    """reference :10-16: scale to `lufs` integrated loudness; unchanged when |loudness| > 100 (silence, near silence)."""
    loudness = integrated_loudness(audio_array, sr)
    if abs(loudness) > 100:
        return audio_array
    gain = 10.0 ** ((lufs - loudness) / 20.0)
    return (np.asarray(audio_array, dtype=np.float64) * gain).astype(np.float32)


def audio_prepare_single(audio_path, sample_rate=16000):
    """reference :67-75 for WAV files: mono, `sample_rate`, loudness-normalised float32."""
    ext = os.path.splitext(audio_path)[1].lower()
    if ext in _VIDEO:
        raise ValueError(f"{audio_path}: audio inside video containers is not decoded here (the reference runs ffmpeg); "
                         f"extract it first: `ffmpeg -i {os.path.basename(audio_path)} -vn -ac 1 -ar {sample_rate} "
                         f"-acodec pcm_s16le out.wav`")
    return loudness_norm(load_audio(audio_path, sample_rate), sample_rate)


def embedding_device(speech_array, wav2vec_feature_extractor, audio_encoder, sr=16000, device=None):
    """The embedding [S, layers, D] f32 left on the GPU (the pipeline keeps it there for the window cut)."""
    seq_len = int(len(speech_array) / sr * 25)                        # video length at 25 fps (reference :19-20, 31)
    values = np.squeeze(wav2vec_feature_extractor(speech_array, sampling_rate=sr).input_values)
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    eng = audio_encoder.engine(dev)
    return eng.forward(torch.from_numpy(np.ascontiguousarray(values, dtype=np.float32)).to(dev), seq_len)


def get_embedding(speech_array, wav2vec_feature_extractor, audio_encoder, sr=16000, device=None):
    """reference :18-41: [S, layers, D] fp32 on the CPU (the encoder itself runs on `device`, default the current GPU)."""
    return embedding_device(speech_array, wav2vec_feature_extractor, audio_encoder, sr, device).cpu()


def cut_windows(audio_embed, num_frames, audio_start_idx=0):
    """[S, layers, D] -> [1, num_frames, 5, layers, D]: frame i gets rows audio_start_idx + i - 2 .. + 2, clamped to
    [0, S - 1] (reference svi_video_talk.py:412-430).  A gather on the tensor's device."""
    idx = torch.arange(audio_start_idx, audio_start_idx + num_frames, device=audio_embed.device)[:, None] + \
        torch.arange(-2, 3, device=audio_embed.device)[None]
    idx = idx.clamp_(0, audio_embed.shape[0] - 1)
    return audio_embed[idx][None]


def cut_audio_embedding(audio_embed, num_frames, audio_start_idx=0, audio_end_idx=81):
    """reference :79-108 (training data path): audio_embed [layers, S, D] ('b s d') -> (first-frame windows [1, 5, layers,
    D], latter-frame windows [(num_frames - 1) / 4, 8, layers, D]) in the layout preprocess_audio produces.
    audio_end_idx is ignored, as in the reference (it is recomputed from num_frames)."""
    from diffsynth.pipelines.svi_video_talk import preprocess_audio
    emb = audio_embed.transpose(0, 1)                                 # "b s d -> s b d"
    first, latter = preprocess_audio(cut_windows(emb, num_frames, audio_start_idx))
    return first.squeeze(0), latter.squeeze(0)
