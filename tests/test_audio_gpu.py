"""GPU: the wav2vec2 audio encoder of SVI-Talk — each new kernel against an fp64 torch computation at the real widths with
ragged lengths, the first convolution's whole-sequence statistics at T0 ~ 2e6, the tiny and the chinese-wav2vec2-base
sized encoder against the oracle, run-to-run reproducibility on 2 minutes of audio, and a clip through
pipe(audio_path=...) against the same pipeline fed the oracle's window features."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import wav2vec2_oracle as O  # noqa: E402
from tools import synth_audio as SA  # noqa: E402

pytestmark = pytest.mark.gpu


def _nv():
    from diffsynth import _native as nv
    return nv


def _rel(got, ref):
    err = (got.double() - ref.double()).abs()
    return err.max().item(), (err.mean() / ref.double().abs().mean()).item()


def _model(cfg, seed=0):
    from utils.src.audio_analysis.wav2vec2 import Wav2Vec2Model
    m = Wav2Vec2Model(cfg)
    m.load_state_dict(SA.make_state_dict(cfg, seed=seed))
    return m.eval()


@pytest.mark.parametrize("n", [16000 * 3 + 7, 4001])
def test_conv0_groupnorm_gelu(n):
    nv = _nv()
    g = torch.Generator().manual_seed(n)
    wav = (0.2 + torch.randn(n, generator=g)).cuda()
    w = (torch.randn(512, 10, generator=g) / 3).cuda()
    gamma, beta = (1 + 0.1 * torch.randn(512, generator=g)).cuda(), (0.1 * torch.randn(512, generator=g)).cuda()
    T0 = (n - 10) // 5 + 1
    out = torch.empty(T0, 512, device="cuda", dtype=torch.bfloat16)
    nv.audio_conv0_gn_gelu(wav, w, gamma, beta, 1e-5, 5, out)
    v = F.conv1d(wav.double()[None, None], w.double()[:, None], stride=5)
    ref = F.gelu(F.group_norm(v, 512, gamma.double(), beta.double(), 1e-5))[0].T
    err = (out.double() - ref).abs()
    print(f"conv0 n={n}: max err {err.max().item():.3e}")
    assert (err <= 2.0 ** -8 * ref.abs() + 1e-3).all()


def test_conv0_statistics_at_two_million_rows():
    nv = _nv()
    n = 5 * 2_000_000 + 9
    g = torch.Generator().manual_seed(7)
    t = torch.arange(n, dtype=torch.float64) / 16000
    wav = (0.3 + 0.5 * torch.sin(2 * torch.pi * 220 * t) + 0.1 * torch.randn(n, generator=g, dtype=torch.float64)).float().cuda()
    w = (torch.randn(512, 10, generator=g) / 3).cuda()
    gamma, beta = torch.ones(512, device="cuda"), torch.zeros(512, device="cuda")
    T0 = (n - 10) // 5 + 1
    out = torch.empty(T0, 512, device="cuda", dtype=torch.bfloat16)
    ws = nv.audio_conv0_gn_gelu(wav, w, gamma, beta, 1e-5, 5, out)
    torch.cuda.synchronize()
    st = ws[:2 * 512 * 4].view(torch.float32)
    mean, rstd = st[:512].double(), st[512:].double()
    v = F.conv1d(wav.double()[None, None], w.double()[:, None], stride=5)[0]
    rm, rv = v.mean(dim=1), v.var(dim=1, unbiased=False)
    rr = 1 / torch.sqrt(rv + 1e-5)
    e_mean = ((mean - rm).abs() / rv.sqrt()).max().item()
    e_rstd = ((rstd - rr).abs() / rr).max().item()
    print(f"conv0 statistics over T0={T0}: max |mean err|/std {e_mean:.2e}, max rel rstd err {e_rstd:.2e}")
    assert e_mean < 1e-6 and e_rstd < 1e-6


@pytest.mark.parametrize("T_in,S", [(499, 250), (137, 71), (3, 1), (100, 200)])
def test_interp_layernorm(T_in, S):
    nv = _nv()
    g = torch.Generator().manual_seed(T_in)
    x = torch.randn(T_in, 512, generator=g).cuda()
    gamma, beta = (1 + 0.1 * torch.randn(512, generator=g)).cuda(), (0.1 * torch.randn(512, generator=g)).cuda()
    out = torch.empty(S, 512, device="cuda", dtype=torch.bfloat16)
    nv.audio_interp_layernorm(x, gamma, beta, 1e-5, out)
    f = F.interpolate(x.double().T[None], size=S, mode="linear", align_corners=True)[0].T
    ref = F.layer_norm(f, (512,), gamma.double(), beta.double(), 1e-5)
    err = (out.double() - ref).abs()
    assert (err <= 2.0 ** -8 * ref.abs() + 1e-4).all(), err.max().item()


@pytest.mark.parametrize("S", [251, 64, 7])
def test_pos_conv(S):
    nv = _nv()
    D, G, K = 768, 16, 128
    g = torch.Generator().manual_seed(S)
    x = torch.randn(S, D, generator=g).cuda()
    w = (torch.randn(D, D // G, K, generator=g) / (D // G * K) ** 0.5).cuda()
    b = (0.1 * torch.randn(D, generator=g)).cuda()
    packed = w.reshape(G, D // G, D // G, K).permute(0, 3, 2, 1).contiguous()
    out = torch.empty_like(x)
    nv.audio_pos_conv(x, packed, b, G, out)
    pos = F.conv1d(x.double().T[None], w.double(), b.double(), padding=K // 2, groups=G)[:, :, :S]
    ref = x.double() + F.gelu(pos)[0].T
    mx, rel = _rel(out, ref)
    print(f"pos conv S={S}: max err {mx:.2e}")
    assert mx < 1e-4


def test_layernorm_f32x2_into_result_slot():
    nv = _nv()
    M, D, L = 203, 768, 12
    x = torch.randn(M, D, device="cuda") * 3 + 1
    gamma, beta = torch.randn(D, device="cuda"), torch.randn(D, device="cuda")
    res = torch.zeros(M, L, D, device="cuda")
    xb = torch.empty(M, D, device="cuda", dtype=torch.bfloat16)
    nv.layernorm_f32x2(x, gamma, beta, 1e-5, res[:, 5], xb)
    ref = F.layer_norm(x.double(), (D,), gamma.double(), beta.double(), 1e-5)
    assert (res[:, 5].double() - ref).abs().max().item() < 1e-4
    assert torch.equal(xb, res[:, 5].to(torch.bfloat16))
    assert res[:, :5].abs().max().item() == 0 and res[:, 6:].abs().max().item() == 0


def test_tiny_encoder_matches_oracle():
    from utils.src.audio_analysis.wav2vec2 import Wav2Vec2FeatureExtractor
    from utils.audio_process import get_embedding
    cfg = SA.W2V_TINY
    G = np.load(os.path.join(ROOT, "tests", "golden", "wav2vec_tiny.npz"))
    got = get_embedding(G["speech"], Wav2Vec2FeatureExtractor(), _model(cfg), device="cuda")
    ref = torch.from_numpy(G["emb"])
    mx, rel = _rel(got, ref)
    print(f"tiny wav2vec2 vs reference golden: max err {mx:.3e}, mean err / mean |ref| {rel:.3e}")
    assert mx < 0.06 and rel < 1.2e-2          # measured on a B200: 3.7e-2, 7.6e-3


def test_base_encoder_10s_matches_oracle():
    from utils.src.audio_analysis.wav2vec2 import Wav2Vec2FeatureExtractor
    from utils.audio_process import get_embedding
    cfg = SA.W2V_BASE
    x = SA.make_waveform(10.013, seed=5)
    sd = SA.make_state_dict(cfg, seed=1)
    m = _model(cfg, seed=1)
    got = get_embedding(x, Wav2Vec2FeatureExtractor(), m, device="cuda")
    torch.set_num_threads(os.cpu_count())
    ref = O.get_embedding(x, sd, cfg)
    assert got.shape == ref.shape == (250, 12, 768)
    mx, rel = _rel(got, ref)
    per_layer = [(got[:, l] - ref[:, l]).abs().max().item() for l in range(12)]
    print(f"base wav2vec2 10 s vs oracle: max err {mx:.3e}, mean err / mean |ref| {rel:.3e}; per layer max "
          + " ".join(f"{e:.3f}" for e in per_layer))
    assert mx < 0.06 and rel < 1.2e-2          # measured on a B200: 3.9e-2, 7.3e-3


def test_two_minutes_finite_and_reproducible():
    from utils.src.audio_analysis.wav2vec2 import Wav2Vec2FeatureExtractor
    from utils.audio_process import embedding_device
    cfg = SA.W2V_BASE
    x = SA.make_waveform(120.0, seed=6)
    m = _model(cfg, seed=1)
    fe = Wav2Vec2FeatureExtractor()
    a = embedding_device(x, fe, m, device="cuda").clone()
    b = embedding_device(x, fe, m, device="cuda")
    assert a.shape == (3000, 12, 768)
    assert torch.isfinite(a).all()
    assert torch.equal(a, b)


def test_talk_clip_from_audio_path(tmp_path):
    """pipe(..., audio_path=<WAV>) against the same pipeline given the oracle's window features as audio_embed=."""
    from scipy.io import wavfile
    from diffsynth import ModelManager, SVITalkVideoPipeline
    from diffsynth.models.wan_video_dit import WanModel
    from diffsynth.models.wan_video_vae import WanVideoVAE
    from test_pipeline_gpu import H, W, _ClipStub, _image, _prompter
    import types
    from tools import synth, synth_vae
    from utils.audio_process import audio_prepare_single
    cfg = synth.CFG_TINY_TALK
    dit = WanModel(**cfg).eval()
    dit.load_state_dict({k: v.to(torch.bfloat16).float() for k, v in synth.make_dit_state_dict(cfg, seed=5).items()})
    vae = WanVideoVAE().eval()
    vae.load_state_dict({k: v.to(torch.bfloat16).float() for k, v in synth_vae.make_vae_state_dict(seed=0).items()})
    mm = ModelManager(torch_dtype=torch.bfloat16, device="cuda")
    mm.add_model("wan_video_dit", dit.to("cuda"))
    mm.add_model("wan_video_vae", vae.to("cuda"))
    w2v_sd = SA.make_state_dict(SA.W2V_BASE, seed=1)
    w2v = SA.write_model_dir(str(tmp_path / "w2v"), SA.W2V_BASE, w2v_sd)
    wav = str(tmp_path / "talk.wav")
    wavfile.write(wav, 16000, (SA.make_waveform(1.9, seed=8) * 32767).astype(np.int16))
    pipe = SVITalkVideoPipeline.from_model_manager(mm, torch_dtype=torch.bfloat16, device="cuda", is_test=True, wav2vec_path=w2v)
    pipe.prompter = _prompter
    pipe.image_encoder = _ClipStub()
    img = _image()
    args = types.SimpleNamespace(ref_pad_cfg=False, ref_pad_num=-1, sequential_cfg="none")
    kw = dict(prompt="p", negative_prompt="n", input_image=img, num_inference_steps=3, cfg_scale={"text": 5.0, "audio": 4.0},
              seed=42, tiled=False, random_ref_frame=torch.from_numpy(np.array(img)), height=H, width=W, num_frames=9, args=args,
              progress_bar_cmd=lambda x: x)
    got = np.stack([np.array(f) for f in pipe(audio_path=wav, audio_start_idx=3, **kw)]).astype(np.float32)
    ref_emb = O.cut_windows(O.get_embedding(audio_prepare_single(wav), w2v_sd, SA.W2V_BASE), 9, 3)
    want = np.stack([np.array(f) for f in pipe(audio_embed=ref_emb, **kw)]).astype(np.float32)
    diff = np.abs(got - want)
    print(f"talk clip audio_path vs oracle features: mean {diff.mean():.3f} levels, p99 {np.percentile(diff, 99):.1f}, "
          f"max {diff.max():.0f}")
    assert diff.mean() < 1.0 and np.percentile(diff, 99) < 5    # measured on a B200: 0.69, 3
