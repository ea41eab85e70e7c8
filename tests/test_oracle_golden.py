"""CPU: the oracle restatement (oracle/) must reproduce the golden vectors produced by the REAL reference
modules (tests/golden/make_golden.py).  This is what pins the oracle; tolerances are fp32 round-off."""
import os

import numpy as np
import pytest
import torch

from oracle import wan_dit_oracle as O
from tools import synth

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    return {k: v for k, v in np.load(os.path.join(GOLD, name + ".npz")).items()}


@pytest.mark.parametrize("name,cfg", [("dit_tiny_t2v", synth.CFG_TINY_T2V), ("dit_tiny_i2v", synth.CFG_TINY_I2V)])
def test_dit_forward_matches_reference(name, cfg):
    g = _load(name)
    f, h, w = (int(v) for v in g["fhw"])
    seed = int(g["seed"])
    sd = synth.make_dit_state_dict(cfg, seed=seed)
    # the synthetic weights must be regenerated bit-identically, otherwise the golden outputs are meaningless
    assert abs(sum(v.double().sum().item() for v in sd.values()) - float(g["weight_checksum"])) < 1e-6
    inp = synth.make_dit_inputs(cfg, f, h, w, seed=seed, ctx_len=int(g["ctx_len"]))
    ts = torch.from_numpy(g["timestep"])
    out = O.dit_forward(sd, cfg, inp["x"], ts, inp["context"], inp.get("clip_feature"), inp.get("y"))
    ref = torch.from_numpy(g["out"])
    assert out.shape == ref.shape
    torch.testing.assert_close(out, ref, rtol=2e-4, atol=2e-4)


@pytest.mark.parametrize("name,cfg", [("dit_tiny_t2v", synth.CFG_TINY_T2V), ("dit_tiny_i2v", synth.CFG_TINY_I2V)])
def test_dit_pieces_match_reference(name, cfg):
    g = _load(name)
    f, h, w = (int(v) for v in g["fhw"])
    seed = int(g["seed"])
    sd = synth.make_dit_state_dict(cfg, seed=seed)
    inp = synth.make_dit_inputs(cfg, f, h, w, seed=seed, ctx_len=int(g["ctx_len"]))
    ts = torch.from_numpy(g["timestep"])
    t, t_mod, ctx = O.embed_conditions(sd, cfg, ts, inp["context"], inp.get("clip_feature"), torch.float32)
    torch.testing.assert_close(t, torch.from_numpy(g["t"]), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(t_mod, torch.from_numpy(g["t_mod"]), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(ctx, torch.from_numpy(g["ctx"]), rtol=1e-4, atol=1e-5)
    ang = O.rope_angles_3d(128, f, h // 2, w // 2)
    blk_x = torch.from_numpy(g["blk_x"])
    torch.testing.assert_close(O.rope_apply(blk_x, ang, cfg["num_heads"]), torch.from_numpy(g["rope_out"]),
                               rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(O.rms_norm(blk_x, sd["blocks.0.self_attn.norm_q.weight"], cfg["eps"]),
                               torch.from_numpy(g["rms_out"]), rtol=1e-5, atol=1e-6)
    blk = O.dit_block(sd, 0, blk_x, ctx, t_mod, ang, cfg)
    torch.testing.assert_close(blk, torch.from_numpy(g["blk_out"]), rtol=1e-4, atol=1e-4)


def test_flow_match_schedule_and_step():
    g = _load("flow_match")
    for steps in (1, 4, 50):
        sig = O.flow_match_sigmas(steps, shift=5.0)
        np.testing.assert_allclose(sig.numpy(), g[f"sigmas_{steps}"], rtol=0, atol=1e-7)
        np.testing.assert_allclose((sig * 1000).numpy(), g[f"timesteps_{steps}"], rtol=0, atol=1e-4)
    sig = O.flow_match_sigmas(4, shift=5.0)
    x = torch.from_numpy(g["step_x"][0])
    for i in range(4):
        x = O.flow_match_step(sig, i, torch.from_numpy(g["step_v"][i]), x)
        np.testing.assert_allclose(x.numpy(), g["step_x"][i + 1], rtol=1e-6, atol=1e-6)
    # documented anchors from the survey (SURVEY.md §8c)
    ts = O.flow_match_sigmas(50, 5.0) * 1000
    assert abs(ts[0].item() - 1000.0) < 1e-3 and abs(ts[1].item() - 995.93) < 1e-2 and abs(ts[-1].item() - 92.59) < 1e-2


def test_flops_formula_matches_survey():
    # SURVEY.md §8(d): cfg-2 283.0 TF, cfg-1 10.35 TF per forward
    assert abs(O.dit_forward_flops(O.CFG_T2V_1_3B, 32760) / 1e12 - 283.0) < 1.0
    assert abs(O.dit_forward_flops(O.CFG_T2V_1_3B, 3200) / 1e12 - 10.35) < 0.1


def _teacache_inputs():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(os.path.dirname(__file__), "golden", "make_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.teacache_inputs()


@pytest.mark.parametrize("model_id", ["Wan2.1-T2V-1.3B", "Wan2.1-I2V-14B-720P"])
@pytest.mark.parametrize("impl", ["oracle", "product"])
def test_teacache_matches_reference_class(model_id, impl):
    """tests/golden/teacache.npz holds decisions, accumulated distances and token streams of the reference's own
    TeaCache class (svi_video.py:23-72) over two back-to-back 12-step clips; both the oracle restatement and the
    product class (its CPU-tensor path: same host logic, torch instead of svi_axpby) must reproduce them."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "teacache.npz"))
    key = model_id.replace(".", "_").replace("-", "_")
    t_mods, xs, outs = _teacache_inputs()
    thresh = float(g[key + "_thresh"])
    if impl == "oracle":
        from oracle.wan_dit_oracle import TeaCacheOracle
        tc = TeaCacheOracle(len(t_mods), thresh, model_id)
        check = lambda x, tm: tc.check(x, tm)
        acc = lambda: tc.acc
    else:
        from diffsynth.pipelines.svi_video import TeaCache
        tc = TeaCache(len(t_mods), rel_l1_thresh=thresh, model_id=model_id)
        check = lambda x, tm: tc.check(None, x, tm)
        acc = lambda: tc.accumulated_rel_l1_distance
    skipped, accs = [], []
    for k in range(2 * len(t_mods)):
        i = k % len(t_mods)
        x = xs[i].clone()
        if check(x, t_mods[i]):
            skipped.append(k)
            x = tc.update(x)
        else:
            x = outs[i].clone()
            tc.store(x)
        accs.append(float(acc()))
        np.testing.assert_allclose(x.numpy(), g[key + "_tokens"][k], rtol=0, atol=1e-6)
    assert skipped == g[key + "_skipped"].tolist() and len(skipped) > 4
    np.testing.assert_allclose(np.array(accs), g[key + "_acc"], rtol=1e-9, atol=1e-12)
    with pytest.raises((ValueError, KeyError)):
        (TeaCacheOracle if impl == "oracle" else TeaCache)(12, 0.3, "no-such-model")


def test_talk_oracle_matches_reference_model():
    """SVI-Talk: AudioProjModel tokens and the enable_multitalk forward (audio cross-attention per latent frame) against
    the reference WanModel (tests/golden/dit_tiny_talk.npz); also preprocess_audio's window selection."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "dit_tiny_talk.npz"))
    cfg = synth.CFG_TINY_TALK
    f, h, w = (int(v) for v in g["fhw"])
    sd = synth.make_dit_state_dict(cfg, seed=int(g["seed"]))
    inp = synth.make_dit_inputs(cfg, f, h, w, seed=int(g["seed"]), ctx_len=int(g["ctx_len"]))
    audio = synth.make_audio_embed(4 * (f - 1) + 1, seed=int(g["seed"]))
    first, latter = O.preprocess_audio(audio)
    assert first.shape == (1, 1, 5, 12, 768) and latter.shape == (1, f - 1, 8, 12, 768)
    # the golden stores the first frame's windows as the (video frame, window) of every selected feature row
    assert abs(audio.double().sum().item() - float(g["audio_checksum"])) < 1e-6
    src = g["first_src"]
    np.testing.assert_array_equal(first[0].numpy(), audio[0].numpy()[src[..., 0], src[..., 1]])
    np.testing.assert_array_equal(latter.numpy(), g["latter"])
    # latent frame 1 = video frames 1..4: frame 1 windows 0..2, frames 2,3 centre window, frame 4 windows 2..4
    assert torch.equal(latter[0, 0, :3], audio[0, 1, :3]) and torch.equal(latter[0, 0, 3], audio[0, 2, 2])
    assert torch.equal(latter[0, 0, 4], audio[0, 3, 2]) and torch.equal(latter[0, 0, 5:], audio[0, 4, 2:])
    tokens = O.audio_proj(sd, first, latter)
    np.testing.assert_allclose(tokens.numpy(), g["audio_tokens"][0], rtol=1e-4, atol=1e-4)
    ts = torch.from_numpy(g["timestep"])
    out = O.dit_forward(sd, cfg, inp["x"], ts, inp["context"], inp["clip_feature"], inp["y"], audio_embed_tuple=(first, latter))
    np.testing.assert_allclose(out.numpy(), g["out"], rtol=2e-4, atol=2e-4)
    base = O.dit_forward(sd, cfg, inp["x"], ts, inp["context"], inp["clip_feature"], inp["y"])
    np.testing.assert_allclose(base.numpy(), g["out_no_audio"], rtol=2e-4, atol=2e-4)
