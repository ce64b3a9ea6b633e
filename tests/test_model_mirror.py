"""The whole-model mirror `visinger_b200.models.visinger.VISinger` against the reference-generated golden
(tests/golden/small_model*.npz, made by tests/golden/make_golden_model.py from the unmodified reference model).

CPU: constructor / state-dict contract and the PyTorch prior network (everything upstream of z_p).
GPU: the full forward(infer=True) waveform in fp32 mode (<= 1e-4) and bf16 / bf16x3 modes."""
import numpy as np
import pytest
import torch

from helpers import load_npz, load_npz_parts, maxabs
from model_inputs import SMALL_HPARAMS, full_hparams, synth_utterances


def _build(precision="fp32"):
    from visinger_b200.models.visinger import VISinger
    z = load_npz_parts("small_model")
    m = VISinger(73, 117, 132, dict(SMALL_HPARAMS), precision=precision).eval()
    sd = {k[2:]: torch.from_numpy(z[k]) for k in z if k.startswith("w/")}
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected
    assert all(k.startswith(("posterior_encoder.", "phoneme_predictor.")) for k in missing)   # training-only modules
    batch = {k[3:]: torch.from_numpy(z[k]) for k in z if k.startswith("in/")}
    return m, z, batch


def test_full_config_state_dict_keys_match_reference_layout():
    """859 entries with the reference's names (checked against the reference in the build container when the golden was
    made); here: spot checks that pin the contract on any box."""
    from visinger_b200.models.visinger import VISinger
    m = VISinger(73, 117, 132, full_hparams())
    sd = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert len(sd) == 859
    assert sd["text_encoder.text_encoder.attn_layers.0.emb_rel_k"] == (1, 9, 96)
    assert sd["text_encoder.embed_positions._float_tensor"] == (1,)
    assert sd["pitch_predictor.pitch_predictor.pre_net.weight"] == (192, 256, 1)
    assert sd["frame_prior.encoder.pre_net.weight"] == (192, 1, 1)
    assert sd["frame_prior.proj.weight"] == (384, 192, 1)
    assert sd["posterior_encoder.pre.weight"] == (192, 1025, 1)
    assert sd["flow.flows.6.enc.in_layers.3.weight_v"] == (384, 192, 5)
    assert sd["decoder.ups.0.weight_g"] == (512, 1, 1)
    assert sd["spk_id_proj.weight"] == (1, 256)
    with pytest.raises(NotImplementedError):
        m(torch.zeros(1, 4, dtype=torch.long), torch.zeros(1, 4, dtype=torch.long), torch.zeros(1, 4, dtype=torch.long),
          torch.ones(1, 8, dtype=torch.long), infer=False)


def test_prior_network_matches_reference_golden():
    m, z, batch = _build()
    ret = {}
    with torch.no_grad():
        mu_p, logs_p, mask, spk = m.prior(batch["text_tokens"], batch["note_pitch"], batch["note_dur"], batch["mel2ph"],
                                          spk_id=batch["spk_ids"], ret=ret)
    assert maxabs(mu_p, torch.from_numpy(z["mu_p"])) <= 2e-5
    assert maxabs(logs_p, torch.from_numpy(z["logs_p"])) <= 2e-5
    assert maxabs(ret["f0_pred"], torch.from_numpy(z["f0_pred"])) <= 2e-5
    assert mask.shape == (3, 1, batch["mel2ph"].shape[1]) and spk.shape == (3, 16, 1)


def test_synthetic_utterance_generator_contract():
    b = synth_utterances(seed=3, n=5, min_frames=120, max_frames=400)
    T = b["mel2ph"].shape[1]
    assert b["text_tokens"].shape == b["note_pitch"].shape == b["note_dur"].shape
    for i in range(5):
        m2p = b["mel2ph"][i]
        n = int((m2p > 0).sum())
        assert 120 <= n <= 400 and bool((m2p[:n] > 0).all()) and bool((m2p[n:] == 0).all())      # right padding only
        assert bool((m2p[1:n] >= m2p[:n - 1]).all()) and int(m2p[0]) == 1                       # monotone, 1-based
        assert int(m2p[:n].max()) == int((b["text_tokens"][i] > 0).sum())                       # every token is used
    assert T == max(int((b["mel2ph"][i] > 0).sum()) for i in range(5))


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16x3", 1e-4), ("bf16", 5e-3)])
def test_full_forward_matches_reference_golden(cuda_device, precision, tol):
    m, z, batch = _build(precision)
    m = m.to(cuda_device)
    d = {k: v.to(cuda_device) for k, v in batch.items()}
    out = m(d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"], spk_id=d["spk_ids"], infer=True,
            noise=torch.from_numpy(z["noise"]).to(cuda_device))
    ref = torch.from_numpy(z["wav_out"])
    assert out["wav_out"].shape == ref.shape                       # [B, T * hop]
    err = maxabs(out["wav_out"].cpu(), ref)
    print(f"full forward {precision}: waveform max-abs err {err:.3e} (|ref|max {float(ref.abs().max()):.3e})")
    assert err <= tol
    # the pitch predictor runs in the path's arithmetic mode too (native RelativeEncoder): fp32 kernels in the parity
    # modes, bf16 tensor-core kernels in the throughput mode (measured 1.04e-2 on log-f0 / uv logits of magnitude ~1)
    assert maxabs(out["f0_pred"].cpu(), torch.from_numpy(z["f0_pred"])) <= (1.6e-2 if precision == "bf16" else 2e-5)


@pytest.mark.gpu
def test_forward_graphed_equals_eager_forward(cuda_device):
    """One CUDA graph per input shape (prior network + hot path) must reproduce the eager forward bit for bit, also
    when it is replayed with different inputs of the same shape."""
    m, z, batch = _build("fp32")
    m = m.to(cuda_device)
    d = {k: v.to(cuda_device) for k, v in batch.items()}
    noise = torch.from_numpy(z["noise"]).to(cuda_device)
    args = (d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"])
    eager = m(*args, spk_id=d["spk_ids"], infer=True, noise=noise)
    got = m.forward_graphed(*args, spk_id=d["spk_ids"], noise=noise)
    assert torch.equal(got["wav_out"], eager["wav_out"]) and torch.equal(got["f0_pred"], eager["f0_pred"])
    noise2 = torch.randn_like(noise)
    eager2 = m(*args, spk_id=d["spk_ids"], infer=True, noise=noise2)
    got2 = m.forward_graphed(*args, spk_id=d["spk_ids"], noise=noise2)          # replay, new contents
    assert torch.equal(got2["wav_out"], eager2["wav_out"])
    assert maxabs(got2["wav_out"].cpu(), torch.from_numpy(z["wav_out"])) > 1e-3     # and it really is a different waveform


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_config4_full_hparams_mixed_length_batch_vs_reference_golden(cuda_device, precision):
    """BASELINE.json configs[3] at the full config/models/visinger.yaml sizes: 8 mixed-length utterances (218 .. 1280
    frames) right-padded to 1280, through the whole forward(infer=True), against the unmodified reference on the
    IDENTICAL padded batch, weights and noise (tests/golden/make_golden_model_full.py) -- strided over the whole waveform,
    the last 20 frames of every utterance in full, and the padded region after each utterance in full (the decoder is
    unmasked, models/visinger.py:111: the reference's output is NOT zero there)."""
    from model_inputs import full_model_mirror, full_model_batch, FULL_GOLDEN_WAV_STRIDE as WS
    z = load_npz("full_model")
    batch, noise, lengths = full_model_batch()
    assert lengths.tolist() == z["lengths"].tolist() and batch["mel2ph"].shape[1] == int(z["T"])
    m = full_model_mirror(precision=precision).to(cuda_device)
    d = {k: v.to(cuda_device) for k, v in batch.items()}
    ret = {}
    out = m(d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"], spk_id=d["spk_ids"], infer=True,
            noise=noise.to(cuda_device))
    wav = out["wav_out"].cpu()
    hop, T = 300, int(z["T"])
    ref_s = torch.from_numpy(z["wav_strided"])
    e_strided = maxabs(wav[:, ::WS], ref_s)
    e_tail = e_pad = 0.0
    for b, n in enumerate(lengths.tolist()):
        e_tail = max(e_tail, maxabs(wav[b, (n - 20) * hop: n * hop], torch.from_numpy(z["wav_tails"][b])))
        seg = wav[b, n * hop: min(T, n + 10) * hop]
        e_pad = max(e_pad, maxabs(seg, torch.from_numpy(z["wav_pads"][b][:seg.numel()])))
    rel = float((wav[:, ::WS] - ref_s).norm() / ref_s.norm())
    e_f0 = maxabs(out["f0_pred"].cpu(), torch.from_numpy(z["f0_pred"]))
    print(f"config 4, full hparams, B=8 mixed lengths, {precision}: waveform max-abs strided {e_strided:.3e}, last 20 frames "
          f"{e_tail:.3e}, padded region {e_pad:.3e} (|ref|max {float(ref_s.abs().max()):.3e}), rel-L2 {rel:.3e}, f0 {e_f0:.3e}")
    if precision == "bf16":
        assert rel <= 3e-2 and max(e_strided, e_tail, e_pad) <= 5e-3
    else:
        assert max(e_strided, e_tail, e_pad) <= 1e-4 and e_f0 <= 5e-5
