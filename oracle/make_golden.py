"""TEST INFRASTRUCTURE: generate tests/golden/*.npz from the RUNNING REFERENCE and pin the oracle.

Run only in the build container (needs /root/reference):   python -m oracle.make_golden
For each case the unmodified reference (through oracle/ref_harness.py's shims) is executed on CPU fp32;
its outputs are (1) compared with oracle/a2p_oracle.py -- the script fails if they disagree -- and
(2) written as the committed fixtures.  The fixtures are the reference's numbers, not the oracle's.
"""
from __future__ import annotations

import hashlib
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import a2p_oracle as O  # noqa: E402
from oracle import ref_harness as RH  # noqa: E402
from oracle.cases import CASES, make_inputs, weights_of, dims_of, layer_inputs  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
TABLES = ["betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod",
          "posterior_variance", "posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2"]


def _close(a, b, what, atol=2e-5, rtol=1e-5):
    """fp32-vs-fp32 noise floor check: tolerances are relative to the output scale max|ref| (CFG with g=10
    amplifies rounding noise ~13x, so face outputs of O(100) carry O(1e-3) absolute fp32 noise)."""
    a, b = a.double(), b.double()
    err = (a - b).abs().max().item()
    scale = max(1.0, b.abs().max().item())
    ok = torch.allclose(a, b, atol=atol * scale, rtol=rtol)
    strict = ((a - b).abs() > 1e-4 + 1e-3 * b.abs()).double().mean().item()
    print(f"   oracle vs reference [{what}]: max|d|={err:.3e} (|ref|max={b.abs().max().item():.3f}; "
          f"outside atol1e-4+rtol1e-3: {100 * strict:.3f}%) {'OK' if ok else 'MISMATCH'}")
    assert ok, what


def golden_schedule():
    ref = RH.import_reference()
    out = {}
    for tag, resp in [("full", ""), ("ddim500", "ddim500"), ("ddim100", "ddim100"), ("ddim10", "ddim10"),
                      ("sec10", "10"), ("sec25_10", "25,10")]:
        args = RH.make_args("pose", 1, 8, resp)
        d = ref.model_util.create_gaussian_diffusion(args)
        o = O.OracleDiffusion(resp)
        out[f"{tag}/timestep_map"] = np.array(d.timestep_map, dtype=np.int64)
        assert list(o.timestep_map) == list(d.timestep_map), tag
        for t in TABLES:
            out[f"{tag}/{t}"] = np.asarray(getattr(d, t), dtype=np.float64)
            if hasattr(o, t):
                assert np.array_equal(getattr(o, t), getattr(d, t)), (tag, t)   # bit-exact
    np.savez_compressed(os.path.join(GOLD, "schedule.npz"), **out)
    print("schedule.npz written; oracle tables bit-identical to reference")


def _ref_model(case, respacing):
    sd = weights_of(case)
    ref, args, model, diffusion = RH.build_reference(case.fmt, case.L, case.H, respacing, sd)
    theirs = {k for k in model.state_dict() if not k.startswith(("audio_model.", "lip_model."))}
    assert theirs == set(sd), theirs ^ set(sd)       # checkpoint key contract == reference
    return ref, model, diffusion, sd


def golden_forward(name):
    case = CASES[name]
    inp = make_inputs(case)
    ref, model, _, sd = _ref_model(case, "ddim10")
    cfg = ref.cfg.ClassifierFreeSampleModel(model)
    y = {"audio": torch.zeros(case.B, 8, 2), "keyframes": inp["keyframes"].clone(), "mask": inp["mask"],
         "scale": inp["scale"]}
    with torch.no_grad(), RH.synthetic_features(model, inp["feats"]):
        c = model(inp["x"], inp["times"], y, cond_drop_prob=0.0)
        u = model(inp["x"], inp["times"], y, cond_drop_prob=1.0)
        g = cfg(inp["x"], inp["times"], y)
    oc = O.denoiser_forward(sd, case.fmt, case.H, inp["x"], inp["times"], inp["feats"], inp["keyframes"], inp["mask"], 0.0)
    ou = O.denoiser_forward(sd, case.fmt, case.H, inp["x"], inp["times"], inp["feats"], inp["keyframes"], inp["mask"], 1.0)
    og = O.cfg_forward(sd, case.fmt, case.H, inp["x"], inp["times"], inp["feats"], inp["keyframes"], inp["mask"], inp["scale"])
    _close(oc, c, name + "/cond"); _close(ou, u, name + "/uncond"); _close(og, g, name + "/cfg", atol=2e-4)
    np.savez_compressed(os.path.join(GOLD, f"fwd_{name}.npz"), cond=c.numpy(), uncond=u.numpy(), cfg=g.numpy(),
                        x_sha1=hashlib.sha1(inp["x"].numpy().tobytes()).hexdigest())
    print(f"fwd_{name}.npz written")


def golden_layer(name):
    """FiLMTransformerDecoderLayer.forward (transformer_modules.py:190-217) of the reference's layer 1 on fixed inputs"""
    case = CASES[name]
    ref, model, _, sd = _ref_model(case, "ddim10")
    x, mem, t, mem2 = layer_inputs(case)
    layer = model.seqTransDecoder.stack[1]
    with torch.no_grad():
        out = layer(x, mem, t, memory2=mem2)
    mine = O.decoder_layer(x, mem, t, mem2, sd, "seqTransDecoder.stack.1", case.H)
    _close(mine, out, name + "/decoder_layer")
    np.savez_compressed(os.path.join(GOLD, f"layer_{name}.npz"), out=out.numpy(),
                        x_sha1=hashlib.sha1(x.numpy().tobytes()).hexdigest())
    print(f"layer_{name}.npz written")


def golden_loop(name, respacing, kind, eta=0.0, check_oracle=True):
    case = CASES[name]
    ref, model, diffusion, sd = _ref_model(case, respacing)
    n = diffusion.num_timesteps
    inp = make_inputs(case, n_noise=n)
    cfg = ref.cfg.ClassifierFreeSampleModel(model)
    y = {"audio": torch.zeros(case.B, 8, 2), "keyframes": inp["keyframes"].clone(), "mask": inp["mask"],
         "scale": inp["scale"]}
    shape = tuple(inp["x"].shape)
    t0 = time.time()
    with torch.no_grad(), RH.synthetic_features(model, inp["feats"]):
        if kind == "ddim":
            tape = list(inp["noise_tape"])
            old = torch.randn_like
            torch.randn_like = lambda x, *a, **k: tape.pop(0)     # explicit per-step noise tape (eta>0)
            try:
                res = diffusion.ddim_sample_loop(cfg, shape, noise=inp["x"], clip_denoised=False, model_kwargs={"y": y},
                                                 eta=eta)
            finally:
                torch.randn_like = old
        else:
            with RH.repaired_p_sample(ref.gd, inp["noise_tape"]):
                res = diffusion.p_sample_loop(cfg, shape, noise=inp["x"], clip_denoised=False, model_kwargs={"y": y})
    print(f"   reference {kind} loop {name}/{respacing or 'full'}: {time.time() - t0:.1f}s")
    tag = f"{kind}_{name}_{respacing or 'full'}" + (f"_eta{eta}" if eta else "")
    np.savez_compressed(os.path.join(GOLD, f"loop_{tag}.npz"), result=res.numpy())
    print(f"loop_{tag}.npz written")
    if not check_oracle:
        return
    t0 = time.time()
    od = O.OracleDiffusion(respacing)
    fn = lambda x, ts: O.cfg_forward(sd, case.fmt, case.H, x, ts, inp["feats"], inp["keyframes"], inp["mask"], inp["scale"])
    if kind == "ddim":
        ores = od.ddim_sample_loop(fn, inp["x"], eta=eta, noise_tape=inp["noise_tape"])
    else:
        ores = od.p_sample_loop(fn, inp["x"], inp["noise_tape"])
    print(f"   oracle {kind} loop {name}/{respacing or 'full'}: {time.time() - t0:.1f}s")
    _close(ores, res, tag, atol=3e-4, rtol=1e-4)


def golden_loop_variants():
    """Sampler keyword variants of the callers' API (SURVEY 8f N4): clip_denoised=True, skip_timesteps, init_image on the
    DDIM loop; const_noise=True + clip + skip (zeros init image) on the repaired ancestral loop
    (gaussian_diffusion.py:305-310,617-632,890-905; upstream-MDM const_noise)."""
    name = "pose_small"
    case = CASES[name]
    out = {}
    for kind, resp, kw in [("ddim", "ddim10", dict(clip_denoised=True, skip_timesteps=3, init_image="randn")),
                           ("ancestral", "10", dict(clip_denoised=True, skip_timesteps=2, init_image=None, const_noise=True))]:
        ref, model, diffusion, sd = _ref_model(case, resp)
        n = diffusion.num_timesteps - kw["skip_timesteps"]
        inp = make_inputs(case, n_noise=n)
        init = None
        if kw["init_image"] == "randn":
            init = 0.5 * torch.from_numpy(np.random.RandomState(77).standard_normal(tuple(inp["x"].shape)).astype(np.float32))
        cfg = ref.cfg.ClassifierFreeSampleModel(model)
        y = {"audio": torch.zeros(case.B, 8, 2), "keyframes": inp["keyframes"].clone(), "mask": inp["mask"], "scale": inp["scale"]}
        shape = tuple(inp["x"].shape)
        fn = lambda x, ts: O.cfg_forward(sd, case.fmt, case.H, x, ts, inp["feats"], inp["keyframes"], inp["mask"], inp["scale"])
        od = O.OracleDiffusion(resp)
        with torch.no_grad(), RH.synthetic_features(model, inp["feats"]):
            if kind == "ddim":
                res = diffusion.ddim_sample_loop(cfg, shape, noise=inp["x"], clip_denoised=True, model_kwargs={"y": y},
                                                 skip_timesteps=kw["skip_timesteps"], init_image=init)
                ores = od.ddim_sample_loop(fn, inp["x"], clip_denoised=True, skip_timesteps=kw["skip_timesteps"], init_image=init)
            else:
                with RH.repaired_p_sample(ref.gd, inp["noise_tape"]):
                    res = diffusion.p_sample_loop(cfg, shape, noise=inp["x"], clip_denoised=True, model_kwargs={"y": y},
                                                  skip_timesteps=kw["skip_timesteps"], const_noise=True)
                ores = od.p_sample_loop(fn, inp["x"], inp["noise_tape"], const_noise=True, clip_denoised=True,
                                        skip_timesteps=kw["skip_timesteps"])
        _close(ores, res, f"variants/{kind}", atol=3e-4, rtol=1e-4)
        out[kind] = res.numpy()
    np.savez_compressed(os.path.join(GOLD, "loop_variants_pose_small.npz"), **out)
    print("loop_variants_pose_small.npz written")


def golden_plms():
    """plms_sample_loop (gaussian_diffusion.py:938-1158), orders 2 and 4, pose_small ddim10 -> loop_plms_pose_small.npz"""
    case = CASES["pose_small"]
    ref, model, diffusion, sd = _ref_model(case, "ddim10")
    inp = make_inputs(case)
    cfg = ref.cfg.ClassifierFreeSampleModel(model)
    y = {"audio": torch.zeros(case.B, 8, 2), "keyframes": inp["keyframes"].clone(), "mask": inp["mask"], "scale": inp["scale"]}
    fn = lambda x, ts: O.cfg_forward(sd, case.fmt, case.H, x, ts, inp["feats"], inp["keyframes"], inp["mask"], inp["scale"])
    od = O.OracleDiffusion("ddim10")
    out = {}
    for order in (2, 4):
        with torch.no_grad(), RH.synthetic_features(model, inp["feats"]):
            res = diffusion.plms_sample_loop(cfg, tuple(inp["x"].shape), noise=inp["x"], clip_denoised=False, model_kwargs={"y": y},
                                             order=order)
        _close(od.plms_sample_loop(fn, inp["x"], order=order), res, f"plms/order{order}", atol=3e-4, rtol=1e-4)
        out[f"order{order}"] = res.numpy()
    np.savez_compressed(os.path.join(GOLD, "loop_plms_pose_small.npz"), **out)
    print("loop_plms_pose_small.npz written")


def golden_caller():
    """The UNMODIFIED caller: sample/generate.py `_setup_model` + `_run_single_diffusion` on CPU with raw audio (the frozen
    extractor runs inside every denoiser call, model/diffusion.py:355-358) -> tests/golden/caller_pose.npz."""
    import tempfile
    from oracle import caller_case as CC
    ref = RH.import_reference()
    import sample.generate as gen
    tmp = tempfile.mkdtemp(prefix="a2p_caller_")
    path = os.path.join(tmp, "model000000.pt")
    CC.write_checkpoint(path)
    args = CC.caller_args(path, "cpu")
    gt, model_kwargs = CC.caller_inputs()
    old_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self          # shim 2 (CPU): model/diffusion.py:321
    old_randn = torch.randn
    first = [CC.initial_noise()]
    try:
        with RH._cwd(ref.scratch):
            model, diffusion = gen._setup_model(args)
        model_kwargs["y"] = {k: v.to(args.device) if torch.is_tensor(v) else v for k, v in model_kwargs["y"].items()}
        torch.randn = lambda *a, **k: first.pop(0) if first else old_randn(*a, **k)   # the loop's initial noise (noise=None)
        sample, audio, keyframes, gt_seq = gen._run_single_diffusion(args, model_kwargs, diffusion, model, CC.inv_transform, gt)
    finally:
        torch.Tensor.cuda = old_cuda
        torch.randn = old_randn
    np.savez_compressed(os.path.join(GOLD, "caller_pose.npz"), sample=sample.numpy(), keyframes=np.asarray(keyframes),
                        gt=gt_seq.numpy(), audio_sha1=hashlib.sha1(np.ascontiguousarray(audio).tobytes()).hexdigest())
    print("caller_pose.npz written", tuple(sample.shape), float(sample.abs().max()))


def golden_guide():
    """The reference's GuideTransformer (logits + KV-free generate under an inverse-CDF draw) and TemporalVertexCodec.decode
    with the seeded weights of oracle/guide_case.py -> tests/golden/guide.npz."""
    from torch.distributions import Categorical
    from oracle import guide_case as GC
    ref = RH.import_reference()
    import model.guide as G
    import model.vqvae as V
    c = GC.GUIDE
    with RH._cwd(ref.scratch):
        m = G.GuideTransformer(tokens=c["tokens"], num_layers=c["layers"], dim=c["dim"], emb_len=798, num_audio_layers=2).eval()
    fixed = {k: m.state_dict()[k].clone() for k in ("rotary.freqs", "audio_resampler.kernel")}
    guide_layout = GC.layout(m.state_dict())
    m.load_state_dict(GC.seeded_state(guide_layout, c["seed"], fixed), strict=True)
    B = c["B"]
    cond = GC.guide_audio(B)
    with torch.no_grad():
        logits = m(GC.guide_tokens(B, c["n"], c["tokens"]), cond)
    draw = GC.inverse_cdf_draw(GC.uniform_tape(B))
    old = Categorical.sample
    Categorical.sample = lambda self, *a, **k: draw(self.probs)
    try:
        tokens = m.generate(cond, sequence_length=4, layers=3, n_sequences=B)
    finally:
        Categorical.sample = old
    v = GC.VQ
    codec = V.TemporalVertexCodec(n_vertices=v["n_vertices"], latent_dim=v["latent_dim"], categories=v["categories"],
                                  residual_depth=v["residual_depth"]).eval()
    vq_layout = GC.layout(codec.state_dict())
    codec.load_state_dict(GC.seeded_state(vq_layout, v["seed"]), strict=True)
    with torch.no_grad():
        decoded = codec.decode(GC.vq_codes())
    np.savez_compressed(os.path.join(GOLD, "guide.npz"), guide_layout=guide_layout, guide_fixed_freqs=fixed["rotary.freqs"].numpy(),
                        guide_fixed_kernel=fixed["audio_resampler.kernel"].numpy(), logits=logits.numpy(), tokens=tokens.numpy(),
                        vq_layout=vq_layout, vq_decoded=decoded.numpy())
    print("guide.npz written", tuple(logits.shape), tuple(tokens.shape), tuple(decoded.shape))


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    os.makedirs(GOLD, exist_ok=True)
    if "guide" in sys.argv:
        golden_guide()
        return
    if "plms" in sys.argv:
        golden_plms()
        return
    if "caller" in sys.argv:
        golden_caller()
        return
    if "variants" in sys.argv:
        golden_loop_variants()
        return
    if "loop1000" in sys.argv:     # the benchmarked configuration: all 1000 steps, B = 4, CFG (minutes of CPU time)
        name = "pose_full_b4_g2" if "g2" in sys.argv else "pose_full_b4"
        golden_loop(name, "", "ddim", check_oracle="--no-oracle" not in sys.argv)
        return
    golden_schedule()
    for n in ["pose_small", "pose_small_h4", "face_small", "pose_full", "face_full"]:
        golden_forward(n)
    for n in ["pose_small", "face_small"]:
        golden_layer(n)
    golden_loop("pose_small", "ddim10", "ddim")
    golden_loop("pose_small", "ddim10", "ddim", eta=0.5)
    golden_loop("pose_small", "ddim100", "ddim")
    golden_loop("pose_small", "10", "ancestral")
    golden_loop("face_small", "ddim10", "ddim")
    golden_loop("face_cfg1", "ddim10", "ddim")
    golden_loop("pose_full", "ddim10", "ddim")


if __name__ == "__main__":
    main()
