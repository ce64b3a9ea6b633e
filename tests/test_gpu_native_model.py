"""The whole model in one library call: `vsg_model_forward` / `VISinger.forward_native` (token front end, speaker
condition, pitch head, seeded prior noise and sinusoidal table on the device, chained with the existing stacks).

CPU: the Philox reference against published known answers, argument errors that need no device, `forward_native`'s
refusal of CPU tensors.  GPU: reference goldens in all three modes, agreement with `VISinger.forward` across every flag
combination, the position table, the noise, CUDA-graph capture, errors with zero launches, the stand-alone C program and a
4600-frame utterance.

Floors measured on a B200 (1000 W power limit, over every flag combination); every gate sits at 1.5-2x its floor:
  against VISinger.forward on the same inputs and noise (the glue's fp32 summation order against cuBLAS / cuDNN):
  fp32 waveform max-abs 8.9e-8 -> gate 1.6e-7; bf16x3 waveform 1.3e-6 -> gate 2.5e-6; f0_pred 6.0e-7 -> gate 1e-6;
  bf16 (the Python glue runs in TF32 there) waveform rel-L2 8.8e-3 -> gate 1.6e-2;
  one 4600-frame utterance, full hparams, bf16: rel-L2 1.2e-2 -> gate 2e-2.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from helpers import load_npz, load_npz_parts, maxabs
from model_inputs import SMALL_HPARAMS, synth_utterances

VSG_EINVAL, VSG_ENOMEM = -1, -3
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ---- Philox4x32-10 reference (numpy) ---------------------------------------------------------------------------------


def philox4x32_10(ctr, key):
    """ctr: uint32 [..., 4], key: uint32 [..., 2] -> uint32 [..., 4] (Salmon et al., SC'11; Random123's philox4x32)."""
    c = [ctr[..., i].astype(np.uint64) for i in range(4)]
    k0, k1 = key[..., 0].astype(np.uint64), key[..., 1].astype(np.uint64)
    M = np.uint64(0xFFFFFFFF)
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(0x9E3779B9)) & M
            k1 = (k1 + np.uint64(0xBB67AE85)) & M
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & M, p1 >> np.uint64(32), p1 & M
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, -1).astype(np.uint32)


def noise_reference(seeds, C, T):
    """The statement of vsg_normal_noise in float64 (before the final rounding to fp32)."""
    s = np.asarray(seeds, dtype=np.uint64)
    b, c, t = np.meshgrid(np.arange(len(s)), np.arange(C), np.arange(T), indexing="ij")
    ctr = np.stack([t, c, np.zeros_like(t), np.zeros_like(t)], -1).astype(np.uint32)
    key = np.stack([s[b] & np.uint64(0xFFFFFFFF), s[b] >> np.uint64(32)], -1).astype(np.uint32)
    x = philox4x32_10(ctr, key)
    u1 = (x[..., 0].astype(np.float64) + 1.0) * 2.0 ** -32
    u2 = x[..., 1].astype(np.float64) * 2.0 ** -32
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def test_philox_reference_known_answers():
    """Random123's published known-answer vectors for philox4x32_10."""
    kat = [([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
           ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
           ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
            [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]
    for ctr, key, want in kat:
        got = philox4x32_10(np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32))
        assert got.tolist() == want


def _small_model(hp_over=None, seed=0, precision="fp32"):
    from visinger_b200.models.visinger import VISinger
    hp = dict(SMALL_HPARAMS)
    hp.update(hp_over or {})
    torch.manual_seed(seed)
    m = VISinger(73, 117, 132, hp, precision=precision).eval()
    with torch.no_grad():       # the reference zero-initialises the flow's `post` (an identity flow): give it weights
        for f in range(4):
            post = m.flow.flows[2 * f].post
            post.weight.normal_(0, 0.05)
            post.bias.normal_(0, 0.05)
    return m


def _cfg(**kw):
    from visinger_b200 import _lib
    c = _lib.VsgModelConfig(73, 117, 132, 32, 64, 2, 9, 4, 2, 2, 2, 1, 1, 1, 0, 2, 0)
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def test_model_calls_reject_bad_arguments_without_gpu():
    from visinger_b200 import _lib
    L = _lib.lib()
    out = ctypes.c_void_p()
    assert L.vsg_model_pack_create(None, None, 0, b"", 0, ctypes.byref(out)) == VSG_EINVAL and not out.value
    # a model without any speaker condition (the reference's speaker_embedding would return the integer 0)
    rc = L.vsg_model_pack_create(ctypes.byref(_cfg(use_spk_id=0)), None, 0, b"", 0, ctypes.byref(out))
    assert rc == VSG_EINVAL and b"speaker" in L.vsg_last_error()
    rc = L.vsg_model_pack_create(ctypes.byref(_cfg()), None, 0, b"", 0, ctypes.byref(out))   # hot config missing
    assert rc == VSG_EINVAL and not out.value
    assert L.vsg_model_workspace_bytes(None, 1, 4, 8, 0) == 0
    args = [None] * 14 + [1, 4, 8, 0, None, 0, None]
    assert L.vsg_model_forward(*args) == VSG_EINVAL and L.vsg_last_launch_count() == 0
    assert L.vsg_normal_noise(None, None, 1, 2, 3, None) == VSG_EINVAL
    assert L.vsg_normal_noise(None, None, -1, 2, 3, None) == VSG_EINVAL
    assert L.vsg_debug_position_table(None, 4, 2, None, None) == VSG_EINVAL


def test_forward_native_refuses_cpu_tensors():
    m = _small_model()
    b = synth_utterances(seed=1, n=2, min_frames=40, max_frames=60)
    with pytest.raises(RuntimeError, match="CPU fallback"):
        m.forward_native(b["text_tokens"], b["note_pitch"], b["note_dur"], b["mel2ph"], spk_id=b["spk_ids"])


# ---- GPU ---------------------------------------------------------------------------------------------------------------


def _to(d, dev):
    return {k: v.to(dev) for k, v in d.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16x3", 1e-4), ("bf16", 5e-3)])
def test_small_golden_through_forward_native(cuda_device, precision, tol):
    """The gates of test_model_mirror.py::test_full_forward_matches_reference_golden."""
    from visinger_b200.models.visinger import VISinger
    z = load_npz_parts("small_model")
    m = VISinger(73, 117, 132, dict(SMALL_HPARAMS), precision=precision).eval()
    m.load_state_dict({k[2:]: torch.from_numpy(z[k]) for k in z if k.startswith("w/")}, strict=False)
    m = m.to(cuda_device)
    d = _to({k[3:]: torch.from_numpy(z[k]) for k in z if k.startswith("in/")}, cuda_device)
    out = m.forward_native(d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"], spk_id=d["spk_ids"],
                           noise=torch.from_numpy(z["noise"]).to(cuda_device))
    ref = torch.from_numpy(z["wav_out"])
    assert out["wav_out"].shape == ref.shape
    err = maxabs(out["wav_out"].cpu(), ref)
    e_f0 = maxabs(out["f0_pred"].cpu(), torch.from_numpy(z["f0_pred"]))
    print(f"forward_native small golden {precision}: waveform max-abs {err:.3e}, f0 {e_f0:.3e}, launches {m.last_launches}")
    assert err <= tol and e_f0 <= (1.6e-2 if precision == "bf16" else 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_full_golden_mixed_lengths_through_forward_native(cuda_device, precision):
    """The comparisons and gates of test_model_mirror.py::test_config4_full_hparams_mixed_length_batch_vs_reference_golden."""
    from model_inputs import full_model_mirror, full_model_batch, FULL_GOLDEN_WAV_STRIDE as WS
    z = load_npz("full_model")
    batch, noise, lengths = full_model_batch()
    m = full_model_mirror(precision=precision).to(cuda_device)
    d = _to(batch, cuda_device)
    out = m.forward_native(d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"], spk_id=d["spk_ids"],
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
    print(f"forward_native full golden {precision}: strided {e_strided:.3e}, tails {e_tail:.3e}, padded {e_pad:.3e}, "
          f"rel-L2 {rel:.3e}, f0 {e_f0:.3e}, launches {m.last_launches}")
    if precision == "bf16":
        assert rel <= 3e-2 and max(e_strided, e_tail, e_pad) <= 5e-3
    else:
        assert max(e_strided, e_tail, e_pad) <= 1e-4 and e_f0 <= 5e-5


# (hparams overrides, speaker inputs, given f0 / uv, utterance lengths)
FLAG_CASES = {
    "pos+pitch+spk_id": (dict(), ("id",), False, None),
    "nopos+pitch+spk_embed": (dict(use_pos_embed=False, use_spk_id=False, use_spk_embed=True), ("embed",), False, None),
    "pos+nopitch+both_spk": (dict(use_pitch_embed=False, use_spk_embed=True), ("id", "embed"), False, None),
    "pos+pitch+both_spk+given_f0": (dict(use_spk_embed=True), ("id", "embed"), True, None),
    "nopos+nopitch+spk_id+given_f0_ignored": (dict(use_pos_embed=False, use_pitch_embed=False), ("id",), True, None),
    "pos_beyond_2000_rows": (dict(), ("id",), False, [2300, 1500]),
}


def _inputs(B_lengths, hp_over, spk, given_f0, dev, seed=5):
    lengths = B_lengths or [170, 120, 90]
    b = synth_utterances(seed=seed, n=len(lengths), lengths=lengths, n_spk=2)
    gen = torch.Generator().manual_seed(seed)
    B, T = b["mel2ph"].shape
    kw = {}
    if "id" in spk:
        kw["spk_id"] = b["spk_ids"].to(dev)
    if "embed" in spk:
        kw["spk_embed"] = torch.randn(B, 256, generator=gen).to(dev)
    if given_f0:
        kw["f0"] = (5.0 + 0.3 * torch.randn(B, T, generator=gen)).to(dev)
        kw["uv"] = (torch.rand(B, T, generator=gen) < 0.3).float().to(dev)
    kw["noise"] = torch.randn(B, 32, T, generator=gen).to(dev)
    args = [b[k].to(dev) for k in ("text_tokens", "note_pitch", "note_dur", "mel2ph")]
    return args, kw


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("case", list(FLAG_CASES))
def test_forward_native_matches_python_forward(cuda_device, case, precision):
    hp_over, spk, given_f0, lengths = FLAG_CASES[case]
    m = _small_model(hp_over, seed=3, precision=precision).to(cuda_device)
    args, kw = _inputs(lengths, hp_over, spk, given_f0, cuda_device)
    ref = m(*args, infer=True, **kw)
    got = m.forward_native(*args, **kw)
    assert set(got) == set(ref)
    w, wr = got["wav_out"].cpu(), ref["wav_out"].cpu()
    e_w, rel = maxabs(w, wr), float((w - wr).norm() / wr.norm())
    e_z = maxabs(got["z_q"].cpu(), ref["z_q"].cpu())
    e_f0 = maxabs(got["f0_pred"].cpu(), ref["f0_pred"].cpu()) if "f0_pred" in ref else 0.0
    print(f"forward_native vs forward [{case}] {precision}: waveform max-abs {e_w:.3e} rel-L2 {rel:.3e}, z_q {e_z:.3e}, "
          f"f0_pred {e_f0:.3e}")
    if precision == "bf16":
        assert rel <= 1.6e-2
    else:
        assert e_w <= (1.6e-7 if precision == "fp32" else 2.5e-6) and e_f0 <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [32, 96, 192, 256])
def test_position_table_against_get_embedding(cuda_device, dim):
    from visinger_b200 import _lib
    from visinger_b200.modules.rel_transformer import SinusoidalPositionalEmbedding
    rows = 30001
    ref = SinusoidalPositionalEmbedding.get_embedding(rows, dim, 0)
    got = _lib.debug_position_table(rows, dim, _lib.position_freq(dim), cuda_device).cpu()
    err = maxabs(got, ref)
    # where torch's fp32 sin / cos are correctly rounded (against float64 numpy), the tables are identical
    freq = _lib.position_freq(dim).numpy()
    ang = (np.arange(rows, dtype=np.float32)[:, None] * freq[None, :]).astype(np.float32).astype(np.float64)
    cr = np.concatenate([np.sin(ang), np.cos(ang)], 1).astype(np.float32)
    cr[0] = 0
    ok = (ref.numpy() == cr).all(1)
    exact = bool((got.numpy()[ok] == cr[ok]).all())
    print(f"position table dim {dim}: max-abs vs get_embedding {err:.3e}, rows with torch correctly rounded "
          f"{int(ok.sum())}/{rows}, identical there: {exact}")
    assert err <= 2.0 ** -24
    assert exact
    # without the frequencies: correctly rounded exp; at most the one-ulp frequency difference away from torch
    fb = _lib.debug_position_table(rows, dim, None, cuda_device).cpu()
    assert maxabs(fb, ref) <= 1.5e-4


@pytest.mark.gpu
def test_normal_noise_statistics_and_batch_independence(cuda_device):
    from scipy import stats
    from visinger_b200 import _lib
    seeds = torch.tensor([12345, 2 ** 63 - 25, 7, 0, 99], dtype=torch.int64)
    C, Tp, T = 40, 300, 517
    alone = _lib.normal_noise(seeds[:1].to(cuda_device), C, Tp).cpu()
    batch = _lib.normal_noise(seeds.to(cuda_device), C, T).cpu()
    assert torch.equal(batch[0, :, :Tp], alone[0])
    ref = noise_reference(seeds.numpy().astype(np.uint64), C, T)
    assert float(np.abs(batch.numpy() - ref).max()) <= 1e-6
    big = _lib.normal_noise(torch.tensor([1, 2], dtype=torch.int64, device=cuda_device), 2, 1000000).cpu().double()
    n = big[0].numel()
    for s in range(2):
        x = big[s].reshape(-1)
        assert abs(float(x.mean())) <= 4 / n ** 0.5
        assert abs(float(x.var()) - 1.0) <= 4 * (2.0 / n) ** 0.5
        p = stats.kstest(x.numpy(), "norm").pvalue
        assert p > 1e-3, p
    r_seed = float(np.corrcoef(big[0].reshape(-1).numpy(), big[1].reshape(-1).numpy())[0, 1])
    r_chan = float(np.corrcoef(big[0, 0].numpy(), big[0, 1].numpy())[0, 1])
    print(f"normal noise: Pearson r between seeds {r_seed:.2e} ({n} pairs), between channels {r_chan:.2e} ({n // 2} pairs)")
    assert abs(r_seed) < 5e-3 and abs(r_chan) < 5e-3


class _Raw:
    """Direct ctypes calls of vsg_model_forward on fixed buffers (what a C caller does)."""

    def __init__(self, m, args, kw, dev, seeds=None):
        from visinger_b200 import _lib
        self.L, self.lib = _lib.lib(), _lib
        self.m = m
        self.pack = m._model_pack(dev)
        self.ints = [a.contiguous() for a in args]
        B, self.T_ph = self.ints[0].shape
        self.B, self.T = B, self.ints[3].shape[1]
        self.spk = kw["spk_id"].cpu().contiguous() if "spk_id" in kw else None
        self.noise = kw.get("noise")
        self.seeds = seeds
        self.prec = _lib.precision_code(m.precision)
        self.wav = torch.empty(B, self.T * self.pack.hop, device=dev)
        self.f0 = torch.empty(B, self.T, 2, device=dev)
        self.zq = torch.empty(B, 32, self.T, device=dev)
        self.need = self.pack.workspace_bytes(B, self.T_ph, self.T, self.prec)
        self.ws = torch.empty(self.need, dtype=torch.uint8, device=dev)
        self.dev = dev

    def __call__(self, ws_bytes=None, **over):
        p = dict(text=self.ints[0].data_ptr(), pitch=self.ints[1].data_ptr(), dur=self.ints[2].data_ptr(),
                 mel2ph=self.ints[3].data_ptr(), spk=self.spk.data_ptr() if self.spk is not None else None, emb=None,
                 f0=None, uv=None, noise=self.noise.data_ptr() if self.noise is not None else None,
                 seeds=self.seeds.data_ptr() if self.seeds is not None else None, wav=self.wav.data_ptr(),
                 f0p=self.f0.data_ptr(), zq=self.zq.data_ptr())
        p.update(over)
        return self.L.vsg_model_forward(self.pack.handle, p["text"], p["pitch"], p["dur"], p["mel2ph"], p["spk"], p["emb"],
                                        p["f0"], p["uv"], p["noise"], p["seeds"], p["wav"], p["f0p"], p["zq"], self.B,
                                        self.T_ph, self.T, self.prec, self.ws.data_ptr(),
                                        self.need if ws_bytes is None else ws_bytes,
                                        torch.cuda.current_stream(self.dev).cuda_stream)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_seeded_call_equals_call_with_drawn_noise(cuda_device, precision):
    from visinger_b200 import _lib
    m = _small_model(seed=4, precision=precision).to(cuda_device)
    args, kw = _inputs(None, {}, ("id",), False, cuda_device)
    seeds = torch.tensor([3, 1 << 40, 77], dtype=torch.int64, device=cuda_device)
    a = m.forward_native(*args, spk_id=kw["spk_id"], seeds=seeds)
    b = m.forward_native(*args, spk_id=kw["spk_id"], noise=_lib.normal_noise(seeds, 32, args[3].shape[1]))
    assert torch.equal(a["wav_out"], b["wav_out"]) and torch.equal(a["z_q"], b["z_q"])


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_model_forward_capture_and_determinism(cuda_device, precision):
    m = _small_model(seed=6, precision=precision).to(cuda_device)
    args, kw = _inputs(None, {}, ("id",), False, cuda_device)
    seeds = torch.tensor([5, 6, 7], dtype=torch.int64, device=cuda_device)
    kw.pop("noise")
    raw = _Raw(m, args, kw, cuda_device, seeds=seeds)
    assert raw() == 0
    eager = raw.wav.clone()
    assert raw() == 0
    assert torch.equal(raw.wav, eager)                       # two eager calls: identical bits
    launches = raw.L.vsg_last_launch_count()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            assert raw() == 0
    torch.cuda.synchronize()
    raw.wav.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(raw.wav, eager)
    # new contents in the same buffers: other tokens (same shapes), other seeds
    args2, _ = _inputs(None, {}, ("id",), False, cuda_device, seed=9)
    Tp, T = raw.T_ph, raw.T
    for dst, src in zip(raw.ints, args2):
        dst.zero_()
        n0, n1 = min(dst.shape[1], src.shape[1]), dst.shape[0]
        dst[:n1, :n0].copy_(src[:n1, :n0])
    seeds.copy_(torch.tensor([50, 60, 70]))
    g.replay()
    torch.cuda.synchronize()
    replayed = raw.wav.clone()
    assert raw() == 0
    torch.cuda.synchronize()
    assert torch.equal(raw.wav, replayed) and not torch.equal(replayed, eager)
    print(f"vsg_model_forward {precision}: {launches} kernel launches per call (B=3, T_ph={Tp}, T={T}); graph replay "
          f"bit-identical to the eager call, also with new inputs")


@pytest.mark.gpu
def test_model_errors_name_the_problem_and_launch_nothing(cuda_device):
    from visinger_b200 import _lib
    m = _small_model(seed=7).to(cuda_device)
    sd = dict(m.state_dict())
    for key in ("text_encoder.linear.bias", "frame_prior.proj.bias", "pitch_predictor.linear.weight"):
        bad = {k: v for k, v in sd.items() if k != key}
        with pytest.raises(RuntimeError) as e:
            _lib.ModelPack(_model_cfg(m), bad, "", cuda_device)
        assert key in str(e.value) and "(-1)" in str(e.value)
    args, kw = _inputs(None, {}, ("id",), False, cuda_device)
    raw = _Raw(m, args, kw, cuda_device)
    L = raw.L
    spk_bad = torch.tensor([0, 2, 1], dtype=torch.int64)
    f0 = torch.zeros(raw.B, raw.T, device=cuda_device)
    cases = {"null text_tokens": dict(text=None), "null wav": dict(wav=None), "spk_id out of range": dict(spk=spk_bad.data_ptr()),
             "missing spk_id": dict(spk=None), "f0 without uv": dict(f0=f0.data_ptr()),
             "noise and seeds both NULL": dict(noise=None, seeds=None),
             "spk_embed on a spk-id model": dict(emb=f0.data_ptr())}
    for what, over in cases.items():
        assert raw() == 0 and L.vsg_last_launch_count() > 0
        rc = raw(**over)
        print(f"{what}: {rc} {L.vsg_last_error().decode()}")
        assert rc == VSG_EINVAL and L.vsg_last_launch_count() == 0, what
    assert raw() == 0
    assert raw(ws_bytes=raw.need - 1) == VSG_ENOMEM and L.vsg_last_launch_count() == 0
    for bad in (dict(text_tokens=args[0].cpu()), dict(mel2ph=args[3][:, None, :]), dict(text_tokens=args[0][:, :-1])):
        a = dict(zip(("text_tokens", "pitch_tokens", "dur_tokens", "mel2ph"), args))
        a.update(bad)
        with pytest.raises(RuntimeError):
            m.forward_native(*a.values(), spk_id=kw["spk_id"], noise=kw["noise"])
    with pytest.raises(RuntimeError):
        m.forward_native(*args, spk_id=kw["spk_id"], noise=kw["noise"][:, :, :-1])
    with pytest.raises(RuntimeError):
        m.forward_native(*args, spk_id=kw["spk_id"], noise=kw["noise"].cpu())


def _model_cfg(m):
    return m._model_pack(next(m.parameters()).device).cfg


@pytest.mark.gpu
def test_c_program_synthesises_what_forward_native_does(cuda_device, tmp_path):
    from visinger_b200 import _lib
    gcc = shutil.which("gcc")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    if gcc is None or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime_api.h")):
        pytest.skip("gcc or the CUDA headers are not available")
    libdir = os.path.dirname(_lib.build())
    cudalib = os.path.join(os.path.dirname(cuda_inc), "lib64")
    exe = str(tmp_path / "vsg_synthesize")
    subprocess.run([gcc, "-O2", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I", cuda_inc,
                    os.path.join(ROOT, "tools", "vsg_synthesize.c"), "-L", libdir, "-lvisinger_b200", "-L", cudalib,
                    "-lcudart", f"-Wl,-rpath,{libdir}", "-o", exe], check=True)
    m = _small_model(seed=8).to(cuda_device)
    args, kw = _inputs(None, {}, ("id",), False, cuda_device)
    seeds = torch.tensor([11, 22, 33], dtype=torch.int64)
    want = m.forward_native(*args, spk_id=kw["spk_id"], seeds=seeds.to(cuda_device))["wav_out"].cpu()
    bundle = tmp_path / "bundle"
    bundle.mkdir()
    (bundle / "config.bin").write_bytes(bytes(_model_cfg(m)))
    off, lines, blobs = 0, [], []
    for k, v in m.state_dict().items():
        v = v.detach().to("cpu", torch.float32).contiguous()
        lines.append(f"{k} {v.dim()} " + " ".join(str(s) for s in v.shape) + f" {off}")
        blobs.append(v.numpy().reshape(-1))
        off += v.numel()
    freq = _lib.position_freq(32)
    lines.append(f"embed_positions.freq 1 {freq.numel()} {off}")
    blobs.append(freq.numpy())
    (bundle / "weights.idx").write_text("\n".join(lines) + "\n")
    (bundle / "weights.bin").write_bytes(np.concatenate(blobs).astype(np.float32).tobytes())
    B, T_ph = args[0].shape
    T = args[3].shape[1]
    ins = [np.array([B, T_ph, T, 0], dtype=np.int64)] + [a.cpu().numpy().reshape(-1) for a in args] + \
          [kw["spk_id"].cpu().numpy(), seeds.numpy()]
    (bundle / "inputs.bin").write_bytes(np.concatenate(ins).astype(np.int64).tobytes())
    out = tmp_path / "wav.f32"
    proc = subprocess.run([exe, str(bundle), str(out)], capture_output=True, text=True)
    print(proc.stdout + proc.stderr)
    assert proc.returncode == 0
    got = torch.from_numpy(np.fromfile(out, dtype=np.float32).reshape(B, -1))
    assert torch.equal(got, want)


@pytest.mark.gpu
def test_long_utterance_full_hparams_bf16(cuda_device):
    """4600 frames: split-key attention in the frame-rate stacks and the chunked length regulator through the one call."""
    from model_inputs import full_model_mirror
    m = full_model_mirror(precision="bf16").to(cuda_device)
    b = synth_utterances(seed=21, n=1, lengths=[4600])
    args = [b[k].to(cuda_device) for k in ("text_tokens", "note_pitch", "note_dur", "mel2ph")]
    noise = torch.randn(1, 192, 4600, generator=torch.Generator().manual_seed(2)).to(cuda_device)
    ref = m(*args, spk_id=b["spk_ids"].to(cuda_device), infer=True, noise=noise)["wav_out"].cpu()
    got = m.forward_native(*args, spk_id=b["spk_ids"].to(cuda_device), noise=noise)["wav_out"].cpu()
    rel = float((got - ref).norm() / ref.norm())
    print(f"forward_native vs forward, 4600 frames, full hparams, bf16: rel-L2 {rel:.3e}, max-abs {maxabs(got, ref):.3e}")
    assert rel <= 2e-2
