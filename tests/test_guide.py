"""N2 / N3 (SURVEY 8f): the KV-cached guide sampler and the VQ decoder against the reference's own modules
(model/guide.py GuideTransformer, model/vqvae.py TemporalVertexCodec) on CPU, with reference-layout checkpoints.
tests/golden/guide.npz holds the reference's outputs for the seeded weights and inputs of oracle/guide_case.py
(oracle/make_golden.py guide).  Host-side PyTorch: no GPU needed."""
import json
import os

import numpy as np
import torch

from oracle import guide_case as GC
from oracle.ref_harness import _StandInWav2Vec


def _golden(golden_dir):
    return np.load(os.path.join(golden_dir, "guide.npz"))


def test_guide_sampler_logits_and_generate_match_reference(golden_dir):
    from audio2photoreal_b200.guide import GuideSampler
    g, c = _golden(golden_dir), GC.GUIDE
    layout = str(g["guide_layout"])
    sd = GC.seeded_state(layout, c["seed"], {"rotary.freqs": g["guide_fixed_freqs"], "audio_resampler.kernel": g["guide_fixed_kernel"]})
    audio_model = _StandInWav2Vec(large=False).eval()            # the frozen extractor the reference's constructor loads
    audio_model.load_state_dict({k[len("audio_model."):]: v for k, v in sd.items() if k.startswith("audio_model.")})
    ours = GuideSampler(sd, tokens=c["tokens"], audio_model=audio_model).eval()
    assert set(ours.state_dict()) == {k for k, _, _ in json.loads(layout)}     # same checkpoint layout, frozen extractor included
    B = c["B"]
    cond = GC.guide_audio(B)
    ref_logits = torch.from_numpy(g["logits"])
    got = ours.logits_for(GC.guide_tokens(B, c["n"], c["tokens"]), cond)
    assert torch.allclose(got, ref_logits, rtol=1e-4, atol=2e-5), (got - ref_logits).abs().max().item()

    # generate(): identical token sequences under the same uniform tape (inverse-CDF draw on both sides)
    got_tok = ours.generate(cond, sequence_length=4, layers=3, n_sequences=B, draw=GC.inverse_cdf_draw(GC.uniform_tape(B)))
    ref_tok = torch.from_numpy(g["tokens"])
    assert got_tok.shape == ref_tok.shape == (B, 12) and torch.equal(got_tok, ref_tok)


def test_vq_decoder_matches_reference_and_checkpoint_layout(golden_dir, tmp_path):
    from audio2photoreal_b200.guide import VQDecoder, setup_tokenizer
    g, v = _golden(golden_dir), GC.VQ
    d = tmp_path / "vq"
    d.mkdir()
    with open(d / "args.json", "w") as f:
        json.dump({"nb_joints": v["n_vertices"], "output_emb_width": v["latent_dim"], "code_dim": v["categories"],
                   "depth": v["residual_depth"]}, f)
    torch.save({"net": GC.seeded_state(str(g["vq_layout"]), v["seed"])}, d / "net_iter.pth")
    ours = setup_tokenizer(str(d / "net_iter.pth"), device="cpu")
    assert isinstance(ours, VQDecoder) and ours.residual_depth == 4 and ours.n_clusters == 32
    want = torch.from_numpy(g["vq_decoded"])
    got = ours.decode(GC.vq_codes())
    assert got.shape == want.shape == (3, 20, 104)
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-6)


def test_results_block_layout(tmp_path):
    """sample/generate.py:146-152,289-292: np.save of a dict with these five keys, re-loadable with allow_pickle"""
    from audio2photoreal_b200.guide import inv_transform, results_block, save_results
    stats = {"pose_mean": np.full(104, 0.1, np.float32), "pose_std_flat": np.float32(0.5), "code_mean": np.zeros(256, np.float32),
             "code_std_flat": np.float32(2.0), "audio_mean": np.zeros(2, np.float32), "audio_std_flat": np.float32(3.0)}
    s = torch.randn(2, 104, 1, 60)
    motion = inv_transform(s.permute(0, 2, 3, 1), "pose", stats).permute(0, 3, 1, 2)
    assert torch.allclose(motion, s * 0.5 + 0.1)
    blk = results_block([motion], [np.zeros((2, 96000, 2), np.float32)], [motion], [torch.full((2,), 60)], [torch.zeros(2, 2, 104)])
    save_results(str(tmp_path / "out" / "results.npy"), blk)
    back = np.load(tmp_path / "out" / "results.npy", allow_pickle=True).item()
    assert set(back) == {"motions", "audio", "gt", "lengths", "keyframes"} and back["motions"].shape == (2, 104, 1, 60)
