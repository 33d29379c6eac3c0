"""The caller: what the reference's `sample/generate.py` functions `_setup_model` and `_run_single_diffusion`
(sample/generate.py:74-97,252-268) do, driven through `audio2photoreal_b200.api.patch_reference()` with RAW y["audio"].

oracle/caller_case.py stands in for the reference checkout under its import names (utils.model_util, model.cfg_sampler,
sample.generate): a caller that makes the same calls with the same arguments, looking up the factories patch_reference()
swaps.  fairseq is not installed anywhere, so the frozen vq-wav2vec is ref_harness's stand-in conv stack, loaded through
`fairseq.checkpoint_utils` exactly where the reference's constructor loads it (model/diffusion.py:140,270-271;
model/utils.py:18-26).  The golden output comes from the UNPATCHED reference's own caller run on CPU
(oracle/make_golden.py caller)."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import caller_case as CC


@pytest.fixture(autouse=True)
def _restore_reference_modules():
    yield
    from audio2photoreal_b200.api import unpatch_reference
    unpatch_reference()


def _patched_generate(monkeypatch, cwd):
    for name, mod in CC.caller_modules().items():
        monkeypatch.setitem(sys.modules, name, mod)
    monkeypatch.chdir(cwd)                      # the constructor resolves ./assets/ against the working directory
    from audio2photoreal_b200.api import patch_reference
    patch_reference()
    return sys.modules["sample.generate"]


def test_setup_model_builds_the_b200_objects_and_fails_loudly_without_gpu(tmp_path, monkeypatch):
    """host side of the drop-in (no GPU needed): the caller's own `_setup_model` constructs Denoiser / CFGDenoiser / Sampler,
    the constructor sets up the frozen extractor like the reference's, a real-layout checkpoint (with audio_model.*) loads,
    and sampling on a CPU device raises instead of falling back."""
    from audio2photoreal_b200 import _lib
    from audio2photoreal_b200.api import CFGDenoiser, Denoiser, Sampler
    gen = _patched_generate(monkeypatch, tmp_path)
    path = str(tmp_path / "model000000.pt")
    CC.write_checkpoint(path)
    args = CC.caller_args(path, "cpu")
    model, diffusion = gen._setup_model(args)
    assert isinstance(model, CFGDenoiser) and isinstance(model.model, Denoiser) and isinstance(diffusion, Sampler)
    assert model.model.audio_model is not None and not model.training
    want = CC.standin_audio_state()
    got = model.model.state_dict()
    for k, v in want.items():
        assert torch.equal(got[k], v), k                       # the checkpoint's frozen extractor was loaded, not stashed
    gt, mk = CC.caller_inputs()
    with pytest.raises(_lib.A2PError):
        gen._run_single_diffusion(args, mk, diffusion, model, CC.inv_transform, gt)


@pytest.mark.gpu
@pytest.mark.parametrize("terms", [0, 2])
def test_unchanged_caller_with_raw_audio_vs_reference_golden(golden_dir, tmp_path, monkeypatch, terms):
    gen = _patched_generate(monkeypatch, tmp_path)
    monkeypatch.setenv("A2P_SPLIT_TERMS", str(terms))
    torch.backends.cudnn.allow_tf32 = False                    # the golden is CPU fp32: keep the frozen conv stack fp32 here too
    torch.backends.cuda.matmul.allow_tf32 = False
    path = str(tmp_path / "model000000.pt")
    CC.write_checkpoint(path)
    args = CC.caller_args(path, "cuda:0")
    gt, mk = CC.caller_inputs()
    model, diffusion = gen._setup_model(args)
    mk["y"] = {k: v.to(args.device) if torch.is_tensor(v) else v for k, v in mk["y"].items()}     # generate.py:131-134
    # the loop draws its initial noise with th.randn(*shape, device=device) (noise=None): CUDA and CPU generators differ, so the
    # test hands the loop the CPU draw the golden run used (test-side only; nothing else in the path is random at eta = 0)
    first = [CC.initial_noise()]
    real_randn = torch.randn

    def randn(*a, **k):
        return first.pop(0).to(k.get("device", "cpu")) if first and tuple(a) == tuple(first[0].shape) else real_randn(*a, **k)
    monkeypatch.setattr(torch, "randn", randn)
    sample, audio, keyframes, gt_seq = gen._run_single_diffusion(args, mk, diffusion, model, CC.inv_transform, gt)
    monkeypatch.setattr(torch, "randn", real_randn)
    assert not first, "the loop did not draw the initial noise through torch.randn"
    g = np.load(os.path.join(golden_dir, "caller_pose.npz"))
    d = (sample.double().cpu() - torch.from_numpy(g["sample"]).double()).abs()
    bad = d > 1e-4 + 1e-3 * torch.from_numpy(g["sample"]).double().abs()
    assert not bad.any(), f"terms={terms}: {bad.double().mean().item():.3%} outside rtol 1e-3/atol 1e-4, max|d|={d.max().item():.3e}"
    assert np.allclose(np.asarray(keyframes.cpu()), g["keyframes"]) and np.allclose(gt_seq.cpu().numpy(), g["gt"])
    assert model.model.launch_count() > 0
