"""Generate golden vectors by running the REAL reference modules (from /root/reference) on CPU.

Runs only in the build container (the reference tree does not exist on the GPU box); its outputs,
``tests/golden/*.npz``, are committed.  The reference ships no tests or golden vectors of its own
(SURVEY.md §4), so these files are what pins the oracle (``oracle/``) to the reference's behaviour.

Import recipe (SURVEY.md §8c): pre-register bare ``diffsynth`` package modules pointing into the reference
tree (skipping its heavy ``__init__``), stub the four missing third-party modules, force the flash-attn
availability flags off so the SDPA branch runs on CPU.

usage:  python tests/golden/make_golden.py [--ref /root/reference]
"""
import argparse
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from tools import synth  # noqa: E402


def import_reference(ref_root):
    def pkg(name, path):
        m = types.ModuleType(name)
        m.__path__ = [path]
        sys.modules[name] = m
        return m

    pkg("diffsynth", os.path.join(ref_root, "diffsynth"))
    pkg("diffsynth.models", os.path.join(ref_root, "diffsynth", "models"))
    pkg("diffsynth.utils", os.path.join(ref_root, "diffsynth", "utils"))
    pkg("diffsynth.schedulers", os.path.join(ref_root, "diffsynth", "schedulers"))

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    class _Any:  # permissive placeholder
        def __init__(self, *a, **k):
            pass

        def __call__(self, *a, **k):
            return None

    stub("xfuser")
    stub("xfuser.core")
    stub("xfuser.core.distributed", get_sequence_parallel_rank=lambda: 0, get_sequence_parallel_world_size=lambda: 1,
         get_sp_group=lambda: None)
    stub("xformers")
    stub("xformers.ops", memory_efficient_attention=None)
    stub("imageio")

    class ModelMixin(torch.nn.Module):
        pass

    class ConfigMixin:
        pass

    stub("diffusers", ModelMixin=ModelMixin, ConfigMixin=ConfigMixin)
    stub("diffusers.configuration_utils", ConfigMixin=ConfigMixin, register_to_config=lambda f: f)
    stub("diffusers.models", ModelMixin=ModelMixin)
    stub("diffusers.models.modeling_utils", ModelMixin=ModelMixin)

    dit = importlib.import_module("diffsynth.models.wan_video_dit")
    dit.FLASH_ATTN_2_AVAILABLE = False
    dit.FLASH_ATTN_3_AVAILABLE = False
    dit.SAGE_ATTN_AVAILABLE = False
    vae = importlib.import_module("diffsynth.models.wan_video_vae")
    fm = importlib.import_module("diffsynth.schedulers.flow_match")
    return dit, vae, fm


def ref_model_fn(dit_mod, model, x, timestep, context, clip_feature=None, y=None):
    """The reference's model_fn_wan_video (svi_video.py:74-137) is a free function in a pipeline module that
    cannot be imported without the whole package; WanModel.forward (wan_video_dit.py:486-567) is its
    documented training twin with identical arithmetic for the non-TeaCache / non-USP path."""
    return model(x, timestep, context, clip_feature=clip_feature, y=y)


def golden_dit(dit_mod, cfg, name, f, h, w, ctx_len, seed):
    model = dit_mod.WanModel(**cfg).eval()
    sd = synth.make_dit_state_dict(cfg, seed=seed)
    missing, unexpected = model.load_state_dict(sd, strict=True), None
    inp = synth.make_dit_inputs(cfg, f, h, w, seed=seed, ctx_len=ctx_len)
    ts = torch.tensor([937.5])
    with torch.no_grad():
        out = ref_model_fn(dit_mod, model, inp["x"], ts, inp["context"], inp.get("clip_feature"), inp.get("y"))
        # intermediate pins: one block, rope, rmsnorm
        blk_x = torch.randn(1, f * (h // 2) * (w // 2), cfg["dim"], generator=torch.Generator().manual_seed(7))
        t = model.time_embedding(dit_mod.sinusoidal_embedding_1d(cfg["freq_dim"], ts))
        t_mod = model.time_projection(t).unflatten(1, (6, cfg["dim"]))
        ctx = model.text_embedding(inp["context"])
        if cfg["has_image_input"]:
            ctx = torch.cat([model.img_emb(inp["clip_feature"]), ctx], dim=1)
        fr = torch.cat([model.freqs[0][:f].view(f, 1, 1, -1).expand(f, h // 2, w // 2, -1),
                        model.freqs[1][:h // 2].view(1, h // 2, 1, -1).expand(f, h // 2, w // 2, -1),
                        model.freqs[2][:w // 2].view(1, 1, w // 2, -1).expand(f, h // 2, w // 2, -1)],
                       dim=-1).reshape(f * (h // 2) * (w // 2), 1, -1)
        blk_out = model.blocks[0](blk_x, ctx, t_mod, fr)
        rope_out = dit_mod.rope_apply(blk_x, fr, cfg["num_heads"])
        rms_out = model.blocks[0].self_attn.norm_q(blk_x)
    np.savez_compressed(os.path.join(HERE, name + ".npz"),
                        out=out.numpy(), timestep=ts.numpy(), blk_x=blk_x.numpy(), blk_out=blk_out.numpy(),
                        rope_out=rope_out.numpy(), rms_out=rms_out.numpy(), t=t.numpy(), t_mod=t_mod.numpy(),
                        ctx=ctx.numpy(), weight_checksum=np.float64(sum(v.double().sum().item() for v in sd.values())),
                        fhw=np.array([f, h, w]), ctx_len=np.int64(ctx_len), seed=np.int64(seed))
    print(name, "out", tuple(out.shape), "std", out.std().item())


def golden_scheduler(fm):
    res = {}
    for steps in (1, 4, 50):
        s = fm.FlowMatchScheduler(shift=5, sigma_min=0.0, extra_one_step=True)
        s.set_timesteps(steps, denoising_strength=1.0, shift=5.0)
        res[f"sigmas_{steps}"] = s.sigmas.numpy()
        res[f"timesteps_{steps}"] = s.timesteps.numpy()
    s = fm.FlowMatchScheduler(shift=5, sigma_min=0.0, extra_one_step=True)
    s.set_timesteps(4, shift=5.0)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 5, generator=g)
    xs = [x.numpy()]
    vs = []
    for i, t in enumerate(s.timesteps):
        v = torch.randn(2, 5, generator=g)
        x = s.step(v, s.timesteps[i], x)
        vs.append(v.numpy())
        xs.append(x.numpy())
    res["step_x"] = np.stack(xs)
    res["step_v"] = np.stack(vs)
    np.savez_compressed(os.path.join(HERE, "flow_match.npz"), **res)
    print("flow_match timesteps_50[:3]", res["timesteps_50"][:3], "last", res["timesteps_50"][-1])


def golden_vae(vae_mod):
    sys.path.insert(0, ROOT)
    from tools import synth_vae
    model = vae_mod.WanVideoVAE().eval()
    sd = synth_vae.make_vae_state_dict(seed=0)
    model.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(11)
    video = torch.rand(3, 9, 32, 48, generator=g) * 2 - 1
    with torch.no_grad():
        lat = model.encode([video], device="cpu")          # [1,16,3,4,6]
        z = torch.randn(1, 16, 3, 4, 6, generator=g)
        dec = model.decode(z, device="cpu")                # [1,3,9,32,48]
    np.savez_compressed(os.path.join(HERE, "vae_tiny.npz"), video=video.numpy(), lat=lat.numpy(), z=z.numpy(),
                        dec=dec.numpy())
    print("vae lat", tuple(lat.shape), "dec", tuple(dec.shape), "dec std", dec.std().item())


def golden_talk(dit_mod):
    """Tiny enable_multitalk WanModel (SVI-Talk): the reference forward with audio window features
    (wan_video_dit.py:486-567 with audio_embed_tuple; AudioProjModel :52-112, SingleStreamMutiAttention models/attention.py).
    xformers is absent here: its memory_efficient_attention ([B, M, H, K] layout, no bias) is replaced by torch SDPA."""
    import torch.nn.functional as F
    att_mod = importlib.import_module("diffsynth.models.attention")

    def mea(q, k, v, attn_bias=None, op=None):
        assert attn_bias is None
        return F.scaled_dot_product_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2)).transpose(1, 2)
    sys.modules["xformers.ops"].memory_efficient_attention = mea
    att_mod.xformers.ops = sys.modules["xformers.ops"]
    from oracle import wan_dit_oracle as O
    cfg = synth.CFG_TINY_TALK
    model = dit_mod.WanModel(**cfg).eval()
    sd = synth.make_dit_state_dict(cfg, seed=5)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all("rope_1d" in k or "norm" in k for k in missing), (missing, unexpected)
    f, h, w = 3, 8, 8
    inp = synth.make_dit_inputs(cfg, f, h, w, seed=5, ctx_len=24)
    audio = synth.make_audio_embed(4 * (f - 1) + 1, seed=5)
    first, latter = O.preprocess_audio(audio)
    ts = torch.tensor([600.0])
    with torch.no_grad():
        tokens = model.audio_proj(first, latter)
        out = model(inp["x"], ts, inp["context"], clip_feature=inp["clip_feature"], y=inp["y"], audio_embed_tuple=(first, latter))
        base = model(inp["x"], ts, inp["context"], clip_feature=inp["clip_feature"], y=inp["y"])
    # the first frame's windows are a gather of the seeded audio features: stored as the (video frame, window) each
    # [12, 768] row comes from, plus a checksum of the features, which keeps the fixture under 1 MB
    feats = audio[0].flatten(2)                 # [video frames, windows, 12 * 768]
    idx = [(feats == r).all(-1).nonzero() for r in first.reshape(-1, feats.shape[-1])]
    assert all(len(i) == 1 for i in idx)
    first_src = torch.cat(idx).reshape(first.shape[1:-2] + (2,)).numpy()
    np.savez_compressed(os.path.join(HERE, "dit_tiny_talk.npz"), out=out.numpy(), out_no_audio=base.numpy(),
                        audio_tokens=tokens.numpy(), first_src=first_src, latter=latter.numpy(),
                        audio_checksum=np.float64(audio.double().sum().item()), fhw=np.array([f, h, w]),
                        seed=np.array(5), ctx_len=np.array(24), timestep=ts.numpy())
    print("talk: out", tuple(out.shape), "audio tokens", tuple(tokens.shape), "max|out - no_audio|", float((out - base).abs().max()))


def golden_encoders():
    """Tiny umT5 text encoder and CLIP visual tower: outputs of the reference modules on seeded weights / inputs."""
    import torchvision.transforms as T
    from tools import synth_enc as SE
    te = importlib.import_module("diffsynth.models.wan_video_text_encoder")
    ie = importlib.import_module("diffsynth.models.wan_video_image_encoder")
    res = {}
    # ---- text encoder (wan_video_text_encoder.py:209-255), per-layer position bias (shared_pos=False), key mask
    cfg = SE.TEXT_TINY
    m = te.WanTextEncoder(shared_pos=False, **cfg).eval()
    m.load_state_dict(SE.make_text_state_dict(cfg, seed=0))
    ids, mask = SE.make_text_inputs(cfg, seq_len=24, valid=17, seed=0)
    with torch.no_grad():
        x0 = m.token_embedding(ids)
        bias0 = m.blocks[0].pos_embedding(ids.shape[1], ids.shape[1])
        blk0 = m.blocks[0](x0, mask, pos_bias=None)
        out = m(ids, mask)
    res.update(text_out=out.numpy(), text_bias0=bias0.numpy(), text_block0=blk0.numpy(), text_ids=ids.numpy(),
               text_mask=mask.numpy())
    # ---- CLIP visual tower through WanImageEncoder.encode_image (wan_video_image_encoder.py:864-880): bicubic resize,
    #      [-1,1] -> [0,1] -> mean/std normalisation, all blocks but the last (use_31_block)
    cfg = SE.CLIP_TINY
    vit = ie.VisionTransformer(pool_type="token", pre_norm=True, post_norm=False, activation="gelu", **cfg).eval()
    sd = {k[len("model.visual."):]: v for k, v in SE.make_clip_state_dict(cfg, seed=0).items()}
    vit.load_state_dict(sd)
    fake = types.SimpleNamespace(model=types.SimpleNamespace(image_size=cfg["image_size"], visual=vit),
                                 transforms=T.Compose([T.Normalize(mean=SE.CLIP_MEAN, std=SE.CLIP_STD)]))
    img = SE.make_clip_image(50, 70, seed=0)
    with torch.no_grad():
        out = ie.WanImageEncoder.encode_image(fake, [img.clone()])
        pre = torch.nn.functional.interpolate(img.clone(), size=(cfg["image_size"],) * 2, mode="bicubic", align_corners=False)
    res.update(clip_out=out.numpy(), clip_resized=pre.numpy())
    np.savez_compressed(os.path.join(HERE, "enc_tiny.npz"), **res)
    print("encoders: text", tuple(res["text_out"].shape), "clip", tuple(res["clip_out"].shape))


def teacache_inputs(steps=12, d=48, L=40, seed=5):
    """Seeded inputs of the TeaCache fixture (shared with the tests): per-step modulation [1,6,d], block-stack input and
    output token streams [1,L,d].  The modulation drifts by ~5 % per step with two jumps, so some steps skip."""
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(1, 6, d, generator=g)
    drift = torch.randn(1, 6, d, generator=g)
    scale = [0.0]
    for k in range(1, steps):
        scale.append(scale[-1] + (0.25 if k in (4, 9) else 0.05))
    t_mods = [base + sc * drift for sc in scale]
    xs = [torch.randn(1, L, d, generator=g) for _ in range(steps)]
    outs = [torch.randn(1, L, d, generator=g) for _ in range(steps)]
    return t_mods, xs, outs


def golden_teacache(ref_root):
    """Runs the reference's own TeaCache class (svi_video.py:23-72).  The pipeline module cannot be imported here
    (it pulls the whole package), so the class definition alone is compiled from the reference file in place —
    nothing is copied into this repository."""
    import ast
    path = os.path.join(ref_root, "diffsynth", "pipelines", "svi_video.py")
    tree = ast.parse(open(path).read())
    node = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "TeaCache"][0]
    ns = {"np": np, "torch": torch, "WanModel": object}
    exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    res = {}
    for model_id, thresh in (("Wan2.1-T2V-1.3B", 0.3), ("Wan2.1-I2V-14B-720P", 0.2)):
        t_mods, xs, outs = teacache_inputs()
        tc = ns["TeaCache"](len(t_mods), rel_l1_thresh=thresh, model_id=model_id)
        skipped, acc, finals = [], [], []
        for k in range(2 * len(t_mods)):               # two clips back to back: the step counter wraps (:60-61)
            i = k % len(t_mods)
            x = xs[i].clone()
            if tc.check(None, x, t_mods[i]):
                skipped.append(k)
                x = tc.update(x)
            else:
                x = outs[i].clone()
                tc.store(x)
            acc.append(float(tc.accumulated_rel_l1_distance))
            finals.append(x.numpy())
        key = model_id.replace(".", "_").replace("-", "_")
        res[key + "_skipped"] = np.array(skipped, dtype=np.int64)
        res[key + "_acc"] = np.array(acc, dtype=np.float64)
        res[key + "_tokens"] = np.stack(finals)
        res[key + "_thresh"] = np.array(thresh)
        print("teacache", model_id, "skipped steps", skipped)
    np.savez_compressed(os.path.join(HERE, "teacache.npz"), **res)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", default="/root/reference")
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    dit_mod, vae_mod, fm = import_reference(a.ref)
    if a.only in ("", "dit"):
        golden_dit(dit_mod, synth.CFG_TINY_T2V, "dit_tiny_t2v", f=3, h=8, w=12, ctx_len=40, seed=0)
        golden_dit(dit_mod, synth.CFG_TINY_I2V, "dit_tiny_i2v", f=2, h=6, w=10, ctx_len=24, seed=1)
    if a.only in ("", "sched"):
        golden_scheduler(fm)
    if a.only in ("", "teacache"):
        golden_teacache(a.ref)
    if a.only in ("", "enc"):
        golden_encoders()
    if a.only in ("", "talk"):
        golden_talk(dit_mod)
    if a.only in ("", "vae") and os.path.exists(os.path.join(ROOT, "tools", "synth_vae.py")):
        golden_vae(vae_mod)
