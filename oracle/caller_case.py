"""TEST INFRASTRUCTURE: the inputs of the "unchanged caller" parity case -- sample/generate.py's `_setup_model` +
`_run_single_diffusion` (sample/generate.py:74-97,252-268) driven with RAW 48 kHz audio, once through the unmodified
reference (oracle/make_golden.py caller -> tests/golden/caller_pose.npz) and once through `patch_reference()` on the GPU.

Everything is regenerated deterministically (numpy RandomState / seeded CPU torch generator) on both sides, so the only
committed artefact is the reference's output.  The checkpoint written here has the layout of a real one: the denoiser's
parameters under the reference's names plus the frozen `audio_model.*` entries (stand-in vq-wav2vec conv stack of the
published geometry, oracle/ref_harness.py shim 1)."""
from __future__ import annotations

import os
from argparse import Namespace

import numpy as np
import torch

from oracle.cases import Case, weights_of

CALLER_CASE = Case("caller_pose", "pose", 2, 8, 2, 160, 531, respacing="ddim10", seed=41, wseed=42)
SEED = 10          # --seed default (utils/diff_parser_utils.py:82)


def standin_audio_state(seed: int = 1234):
    """state_dict entries `audio_model.*` of the stand-in extractor, deterministic (CPU generator)."""
    from oracle.ref_harness import _StandInWav2Vec
    rng = torch.random.get_rng_state()
    torch.manual_seed(seed)
    m = _StandInWav2Vec(large=False)
    torch.random.set_rng_state(rng)
    return {"audio_model." + k: v.detach().clone() for k, v in m.state_dict().items()}


def write_checkpoint(path: str) -> None:
    sd = dict(weights_of(CALLER_CASE))
    sd.update(standin_audio_state())
    torch.save(sd, path)


def caller_args(model_path: str, device) -> Namespace:
    """the fields sample/generate.py and utils/model_util.py read (utils/diff_parser_utils.py generate_args)"""
    c = CALLER_CASE
    return Namespace(data_format="pose", add_frame_cond=1, max_seq_length=600, layers=c.L, heads=c.H, not_rotary=False,
                     unconstrained=False, device=device, timestep_respacing=c.respacing, noise_schedule="cosine", sigma_small=True,
                     lambda_vel=0.0, model_path=model_path, resume_trans=None, guidance_param=c.guidance, batch_size=c.B,
                     num_samples=c.B, num_repetitions=1, curr_seq_length=c.T, seed=SEED, save_dir=os.path.dirname(model_path))


def caller_inputs():
    """(gt [B,C,1,T], model_kwargs) as the collate produces them (data_loaders/tensors.py:33-86) + y.scale (generate.py:128-130)"""
    c = CALLER_CASE
    rs = np.random.RandomState(2000 + c.seed)
    f32 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32))
    y = {
        "audio": f32(0.1 * rs.standard_normal((c.B, c.T * 1600, 2))),
        "keyframes": f32(rs.standard_normal((c.B, len(range(0, c.T, 30)), 104))),
        "mask": torch.ones(c.B, 1, 1, c.T, dtype=torch.bool),
        "lengths": torch.full((c.B,), c.T, dtype=torch.int64),
        "scale": torch.full((c.B,), c.guidance),
    }
    gt = f32(rs.standard_normal((c.B, 104, 1, c.T)))
    return gt, {"y": y}


def initial_noise():
    """what `th.randn(*shape, device=device)` (gaussian_diffusion.py:887-892, noise=None) returns on CPU after fixseed(SEED)"""
    c = CALLER_CASE
    g = torch.Generator().manual_seed(SEED)
    return torch.randn(c.B, 104, 1, c.T, generator=g)


def inv_transform(data, data_type: str):
    """stand-in for Social.inv_transform (data_loaders/data.py:71-91): de-normalise with fixed synthetic statistics"""
    std, mean = {"pose": (0.5, 0.1), "face": (0.7, -0.2), "audio": (2.0, 0.3)}[data_type]
    return data * std + mean


def caller_modules() -> dict:
    """{import name: module} standing in for the reference checkout on sys.path: the module attributes
    `patch_reference()` swaps (the originals raise, so an unswapped one is caught) and a caller that makes the calls of
    sample/generate.py `_setup_model` and `_run_single_diffusion` (:74-107, :252-268) with the same arguments, looking
    the factories up in its module at call time as the original does, plus the stand-in fairseq the model's
    constructor loads the frozen extractor through (model/utils.py:18-26)."""
    import types

    from oracle.ref_harness import fairseq_standin_modules

    def unswapped(*a, **k):
        raise AssertionError("patch_reference() left the reference's own factory in place")
    mods = {n: types.ModuleType(n) for n in ("utils", "utils.model_util", "model", "model.cfg_sampler", "sample", "sample.generate")}
    mu, cs, gen = mods["utils.model_util"], mods["model.cfg_sampler"], mods["sample.generate"]
    mu.create_model_and_diffusion = mu.load_model = mu.create_gaussian_diffusion = unswapped
    cs.ClassifierFreeSampleModel = gen.ClassifierFreeSampleModel = unswapped
    gen.create_model_and_diffusion = gen.load_model = unswapped
    mods["utils"].model_util, mods["model"].cfg_sampler, mods["sample"].generate = mu, cs, gen

    def _setup_model(args):
        model, diffusion = gen.create_model_and_diffusion(args, split_type="test")
        gen.load_model(model, torch.load(args.model_path, map_location="cpu"))
        if args.guidance_param != 1:
            model = gen.ClassifierFreeSampleModel(model)
        model.to(args.device)
        model.eval()
        return model, diffusion

    def _run_single_diffusion(args, model_kwargs, diffusion, model, inv_transform, gt):
        with torch.no_grad():
            sample = diffusion.ddim_sample_loop(model, (args.batch_size, model.nfeats, 1, args.curr_seq_length), clip_denoised=False,
                                                model_kwargs=model_kwargs, init_image=None, progress=True, dump_steps=None,
                                                noise=None, const_noise=False)
        to_frames = lambda t: inv_transform(t.cpu().permute(0, 2, 3, 1), args.data_format).permute(0, 3, 1, 2)
        return (to_frames(sample), inv_transform(model_kwargs["y"]["audio"].cpu().numpy(), "audio"),
                inv_transform(model_kwargs["y"]["keyframes"], args.data_format), to_frames(gt))
    gen._setup_model, gen._run_single_diffusion = _setup_model, _run_single_diffusion
    mods.update(fairseq_standin_modules())
    return mods
