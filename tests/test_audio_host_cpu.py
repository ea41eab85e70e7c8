"""Host logic of the SVI-Talk audio path on the CPU: WAV decoding, BS.1770 loudness, feature normalisation, the checkpoint
loader, the wav2vec2 engine's operation order on torch stand-ins of its kernels, the window cut and the pipeline's
embedding cache.  The stand-ins below restate what each new kernel computes (include/svi_b200.h), rounding to bf16 where
the kernel stores bf16; the GEMM / cast stand-ins come from tests/nv_emulation.py."""
import os
import struct
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "stable-video-infinity_b200"))
from oracle import wav2vec2_oracle as O  # noqa: E402
from tools import synth_audio as SA  # noqa: E402
from utils import audio_process as AP  # noqa: E402
from utils.src.audio_analysis import wav2vec2 as W  # noqa: E402

CFG = SA.W2V_TINY


# ------------------------------------------------------------------------------------------------ kernel stand-ins
def audio_conv0_gn_gelu(wav, w, gamma, beta, eps, stride, out, workspace=None):
    v = F.conv1d(wav.double().reshape(1, 1, -1), w.double()[:, None], stride=stride)
    v = F.group_norm(v, v.shape[1], gamma.double(), beta.double(), eps)
    out.copy_(F.gelu(v)[0].T.to(out.dtype))
    return workspace


def audio_interp_layernorm(x, gamma, beta, eps, out):
    f = F.interpolate(x.T[None], size=out.shape[0], mode="linear", align_corners=True)[0].T
    out.copy_(F.layer_norm(f, f.shape[-1:], gamma, beta, eps).to(out.dtype))
    return out


def audio_pos_conv(x, w_packed, bias, groups, out):
    g, k, cg, _ = w_packed.shape
    w = w_packed.permute(0, 3, 2, 1).reshape(g * cg, cg, k)            # [g][j][c][o] -> [g*cg + o, c, j]
    pos = F.conv1d(x.T[None], w, bias, padding=k // 2, groups=groups)[:, :, :x.shape[0]]
    out.copy_(x + F.gelu(pos)[0].T)
    return out


def layernorm_f32x2(x, gamma, beta, eps, out, out_bf16):
    y = F.layer_norm(x, x.shape[-1:], gamma, beta, eps)
    out.copy_(y)
    out_bf16.copy_(y.to(torch.bfloat16))
    return out


def attention_small(q, k, v, out, num_heads, head_dim, scale, bias_table=None, bucket=None, key_mask=None):
    L = q.shape[0]
    sh = lambda t: t.float().reshape(t.shape[0], num_heads, head_dim).transpose(0, 1)
    a = torch.softmax(sh(q) @ sh(k).transpose(1, 2) * scale, dim=-1) @ sh(v)
    out.copy_(a.transpose(0, 1).reshape(L, -1).to(out.dtype))
    return out


@pytest.fixture
def stand_ins(monkeypatch):
    import nv_emulation
    from diffsynth import _native as nv
    nv_emulation.install(monkeypatch)
    for f in (audio_conv0_gn_gelu, audio_interp_layernorm, audio_pos_conv, layernorm_f32x2, attention_small):
        monkeypatch.setattr(nv, f.__name__, f)


# ------------------------------------------------------------------------------------------------ WAV decoding
def _write_wav24(path, samples, rate, channels):
    data = b"".join(int(s).to_bytes(3, "little", signed=True) for s in samples.reshape(-1))
    fmt = struct.pack("<HHIIHH", 1, channels, rate, rate * channels * 3, channels * 3, 24)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def test_wav_sample_formats(tmp_path):
    from scipy.io import wavfile
    ref = np.array([0.0, 0.5, -0.5, 0.25, -1.0, 0.75], dtype=np.float64)
    cases = {
        "i16": (np.round(ref * 32767).astype(np.int16), lambda d: d / 32768.0),
        "i32": (np.round(ref * 2147483647).astype(np.int32), lambda d: d / 2147483648.0),
        "u8": (np.round(ref * 127 + 128).astype(np.uint8), lambda d: (d.astype(np.float64) - 128) / 128.0),
        "f32": (ref.astype(np.float32), lambda d: d),
    }
    for name, (data, expect) in cases.items():
        p = str(tmp_path / f"{name}.wav")
        wavfile.write(p, 16000, data)
        x, rate = AP.read_wav(p)
        assert rate == 16000 and x.dtype == np.float32
        np.testing.assert_allclose(x, expect(data).astype(np.float32), atol=1e-7, err_msg=name)
    p = str(tmp_path / "i24.wav")
    i24 = np.round(ref * 8388607).astype(np.int64)
    _write_wav24(p, i24, 16000, 1)
    x, _ = AP.read_wav(p)
    np.testing.assert_allclose(x, i24 / 8388608.0, atol=1e-7)


def test_wav_stereo_is_mixed_by_mean_and_resampled(tmp_path):
    from scipy.io import wavfile
    rng = np.random.default_rng(0)
    st = rng.uniform(-0.5, 0.5, size=(4800, 2)).astype(np.float32)
    p = str(tmp_path / "st.wav")
    wavfile.write(p, 16000, st)
    x, _ = AP.read_wav(p)
    np.testing.assert_allclose(x, st.mean(axis=1), atol=1e-7)
    wavfile.write(p, 48000, st)
    y = AP.load_audio(p, 16000)
    assert y.dtype == np.float32 and len(y) == 1600


def test_non_wav_input_names_ffmpeg(tmp_path):
    for name in ("a.mp4", "a.mp3", "a.flac"):
        with pytest.raises(ValueError, match="ffmpeg"):
            AP.audio_prepare_single(str(tmp_path / name))


# ------------------------------------------------------------------------------------------------ BS.1770
def _sine(f, seconds, rate, amp=1.0):
    t = np.arange(int(seconds * rate)) / rate
    return (amp * np.sin(2 * np.pi * f * t)).astype(np.float32)


@pytest.mark.parametrize("rate", [48000, 16000])
def test_full_scale_997hz_sine_reads_minus_3_01_lufs(rate):
    assert abs(AP.integrated_loudness(_sine(997, 5.0, rate), rate) - (-3.01)) < 0.05


def test_gating():
    rate = 16000
    loud = _sine(997, 5.0, rate, 10 ** (-20 / 20))
    alone = AP.integrated_loudness(loud, rate)
    # a 25 dB quieter passage lies below the relative gate (-10 LU); ungated it would pull the result down by ~3 LU.  Only
    # the three blocks straddling the edge (3/4, 1/2, 1/4 loud) are kept: mean energy (47 + 1.5) / 50 of the loud part
    edge = 10 * np.log10(48.5 / 50)
    quiet = _sine(997, 5.0, rate, 10 ** (-45 / 20))
    assert abs(AP.integrated_loudness(np.concatenate([loud, quiet]), rate) - (alone + edge)) < 0.02
    # blocks below -70 LUFS are dropped by the absolute gate
    assert abs(AP.integrated_loudness(np.concatenate([loud, _sine(997, 5.0, rate, 1e-5)]), rate) - (alone + edge)) < 0.02
    silence = np.zeros(rate * 2, dtype=np.float32)
    assert AP.integrated_loudness(silence, rate) == float("-inf")
    np.testing.assert_array_equal(AP.loudness_norm(silence, rate), silence)   # |loudness| > 100: passthrough
    y = AP.loudness_norm(loud, rate)
    assert abs(AP.integrated_loudness(y, rate) - (-23.0)) < 1e-6


def test_feature_normalisation_matches_transformers():
    tr = pytest.importorskip("transformers")
    x = SA.make_waveform(1.3, seed=3)
    ours = W.Wav2Vec2FeatureExtractor(do_normalize=True)(x, sampling_rate=16000).input_values[0]
    ref = np.squeeze(tr.Wav2Vec2FeatureExtractor(do_normalize=True)(x, sampling_rate=16000).input_values)
    np.testing.assert_array_equal(ours, ref)
    np.testing.assert_array_equal(ours, O.feature_normalize(x))


def test_loudness_gain_below_bf16_rounding():
    """+-1 dB of loudness gain (what a different K-weighting design could cost at most) moves the embedding by less than
    the bf16 rounding of its values: the feature extractor's normalisation divides the gain out."""
    sd = SA.make_state_dict(CFG, seed=0)
    x = AP.loudness_norm(SA.make_waveform(1.5, seed=2), 16000)
    base = O.get_embedding(x, sd, CFG)
    for db in (-1.0, 1.0):
        e = O.get_embedding((x * 10 ** (db / 20)).astype(np.float32), sd, CFG)
        assert (e - base).abs().max() < 2.0 ** -9 * base.abs().max()


# ------------------------------------------------------------------------------------------------ checkpoint loader
@pytest.mark.parametrize("spelling,prefix,fmt", [("weight_g", "", "safetensors"), ("parametrizations", "", "bin"),
                                                 ("parametrizations", "wav2vec2.", "safetensors")])
def test_checkpoint_loader(tmp_path, spelling, prefix, fmt):
    sd = SA.make_state_dict(CFG, seed=4)
    D = CFG["hidden_size"]
    extra = {}
    if prefix:                                  # a pre-training checkpoint: quantizer, projections, mask embedding, head
        extra = {"quantizer.codevectors": torch.zeros(1, 8, 4), "quantizer.weight_proj.weight": torch.zeros(8, 32),
                 "project_q.weight": torch.zeros(4, 4), "project_hid.weight": torch.zeros(4, D),
                 "wav2vec2.masked_spec_embed": torch.zeros(D)}
    path = SA.write_model_dir(str(tmp_path / "w2v"), CFG, sd, spelling=spelling, prefix=prefix, extra=extra, fmt=fmt)
    m = W.Wav2Vec2Model.from_pretrained(path, local_files_only=True)
    got = m.state_dict()
    assert set(got) == set(sd)
    for k, v in sd.items():
        torch.testing.assert_close(got[k], v, rtol=0, atol=0)
    fe = W.Wav2Vec2FeatureExtractor.from_pretrained(path)
    assert fe.do_normalize and fe.sampling_rate == 16000


def test_unsupported_config_raises():
    for k, v in (("feat_extract_norm", "layer"), ("do_stable_layer_norm", True), ("conv_bias", True), ("hidden_act", "relu")):
        with pytest.raises(ValueError, match=k):
            W.Wav2Vec2Model(dict(CFG, **{k: v}))


def test_engine_requires_cuda():
    m = W.Wav2Vec2Model(CFG)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.engine("cpu")


# ------------------------------------------------------------------------------------------------ engine on stand-ins
def _model(seed=0):
    m = W.Wav2Vec2Model(CFG)
    m.load_state_dict(SA.make_state_dict(CFG, seed=seed))
    return m.eval()


def test_engine_matches_oracle(stand_ins):
    sd = SA.make_state_dict(CFG, seed=0)
    x = SA.make_waveform(2.0077, seed=1)
    ref = O.get_embedding(x, sd, CFG)
    fe = W.Wav2Vec2FeatureExtractor()
    got = AP.get_embedding(x, fe, _model(), device="cpu")
    assert got.shape == ref.shape == (50, CFG["num_hidden_layers"], CFG["hidden_size"])
    err = (got - ref).abs().max().item()
    print(f"tiny engine on stand-ins vs oracle: max |err| {err:.3e}, max |ref| {ref.abs().max().item():.3f}")
    assert err < 0.08
    # forward() returns all hidden states, hidden_states[1:] being the embedding
    iv = torch.from_numpy(fe(x).input_values[0])[None]
    hs = _model().forward(iv, 50, device="cpu").hidden_states
    assert len(hs) == CFG["num_hidden_layers"] + 1
    torch.testing.assert_close(torch.stack(hs[1:], dim=2)[0], got, rtol=0, atol=0)


def test_window_cut_matches_oracle():
    emb = torch.randn(37, 2, 8)
    for start in (0, 1, 20, 33, 40):
        torch.testing.assert_close(AP.cut_windows(emb, 13, start), O.cut_windows(emb, 13, start), rtol=0, atol=0)


def test_pipeline_caches_the_file_embedding(stand_ins, tmp_path):
    from scipy.io import wavfile
    from diffsynth.pipelines.svi_video_talk import SVITalkVideoPipeline
    sd = SA.make_state_dict(CFG, seed=0)
    path = SA.write_model_dir(str(tmp_path / "w2v"), CFG, sd)
    wav = str(tmp_path / "talk.wav")
    wavfile.write(wav, 16000, (SA.make_waveform(2.0077, seed=1) * 32767).astype(np.int16))
    pipe = SVITalkVideoPipeline(device="cpu", wav2vec_path=path)
    assert pipe.audio_encoder is None                               # nothing loads until the first call
    a = pipe.get_audio_embedding(wav, 13, audio_start_idx=0)
    eng = pipe.audio_encoder.engine("cpu")
    n = eng.launches
    assert n > 0
    b = pipe.get_audio_embedding(wav, 13, audio_start_idx=40)
    assert eng.launches == n                                        # second clip: no encoder launch
    ref = O.get_embedding(AP.audio_prepare_single(wav), sd, CFG)
    assert a.shape == (1, 13, 5, CFG["num_hidden_layers"], CFG["hidden_size"])
    assert (a - O.cut_windows(ref, 13, 0)).abs().max() < 0.08
    assert (b - O.cut_windows(ref, 13, 40)).abs().max() < 0.08
    torch.testing.assert_close(b, AP.cut_windows(pipe.audio_embedding(wav), 13, 40), rtol=0, atol=0)


def test_pipeline_missing_wav2vec_dir(tmp_path):
    from diffsynth.pipelines.svi_video_talk import SVITalkVideoPipeline
    pipe = SVITalkVideoPipeline(device="cpu", wav2vec_path=str(tmp_path / "nope"))
    wav = str(tmp_path / "x.wav")
    from scipy.io import wavfile
    wavfile.write(wav, 16000, np.zeros(16000, dtype=np.int16))
    with pytest.raises(FileNotFoundError, match="nope"):
        pipe.get_audio_embedding(wav, 5)
