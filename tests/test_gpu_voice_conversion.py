"""Voice conversion in one library call: `vsg_spectrogram` / `vsg_model_convert` (VISinger.spectrogram /
VISinger.voice_conversion), on the GPU.

- The spectrogram against the float64 statement (tests/vc_reference.py), every gate relative to S = sum_n |w[n] y[n]| of
  the frame: fp32 / bf16x3 (FFMA, fp32 basis) against the exact value; bf16 (tcgen05) against the statement evaluated on
  the bf16 operands the kernel multiplies (within half a bf16 ulp of the output, which is rounded to bf16, plus a small
  accumulation-order term) and against the exact value within the derived 2^-7 S.  Small config (n_fft 64, hop 15, win 60
  and 64) and full config (2048 / 1200 / 300), T = 1 .. 1000, ragged lengths down to one frame; first and last frames
  are checked on their own.
- Bit-exact equalities: an utterance alone and inside a ragged padded batch (spectrogram and z_hat); the one call against
  the chain vsg_spectrogram -> vsg_posterior_forward -> vsg_flow_forward(reverse=0) -> vsg_infer_zp in all three modes,
  from wav and from spec; a CUDA-graph replay against the eager call; vsg_model_forward on a convert pack against a model
  pack.
- Against the CPU oracle composition (posterior, flow both ways, generator) at the small config (2 speakers, source !=
  target) and the full config (B2 x T400, 4 speakers), all modes.
- Argument errors with zero launches.

Floors measured on a B200 (1000 W power limit); gates at about 2x:
  spectrogram fp32 / bf16x3 against float64: 1.06e-6 S -> gate 2.5e-6 S;
  spectrogram bf16 against the bf16-operand statement, beyond half a bf16 ulp: 2.1e-8 S -> gate 5e-8 S; against the exact
  value 3.9e-3 S -> gate 2^-7 S (the derived bound); the torch.stft statement, rel-L2: fp32 5.0e-7 -> 1e-6, bf16 2.2e-3
  -> 4.5e-3;
  against the oracle composition, waveform: fp32 max-abs 7.5e-8 -> 1.5e-7; bf16x3 max-abs 1.6e-6 -> 3e-6; bf16 rel-L2
  6.5e-3 -> 1.3e-2.
"""
import ctypes

import numpy as np
import pytest
import torch

from helpers import maxabs
from model_inputs import SMALL_HPARAMS, full_hparams
from vc_reference import direct_spectrogram, linear_spectrogram, voice_conversion

pytestmark = pytest.mark.gpu

VSG_EINVAL, VSG_ENOMEM = -1, -3
PREC = {"fp32": 0, "bf16": 1, "bf16x3": 2}


def _model(hp_over=None, full=False, seed=0, precision="fp32"):
    from visinger_b200.models.visinger import VISinger
    hp = full_hparams() if full else dict(SMALL_HPARAMS)
    hp.update(hp_over or {})
    torch.manual_seed(seed)
    m = VISinger(73, 117, 132, hp, precision=precision).eval()
    with torch.no_grad():   # the reference zero-initialises the flow's `post` (an identity flow): give it weights
        for f in range(4):
            post = m.flow.flows[2 * f].post
            post.weight.normal_(0, 0.05)
            post.bias.normal_(0, 0.05)
    return m


def _wav(seed, B, L):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(L, dtype=torch.float64)
    f = 0.005 + 0.3 * torch.rand(B, 1, generator=g, dtype=torch.float64)
    return (0.4 * torch.sin(f * t) + 0.2 * torch.sin(3.1 * f * t + 1.0) +
            0.05 * torch.randn(B, L, generator=g, dtype=torch.float64)).float()


SPEC_CASES = {   # name: (full config, win_size, T, lengths)
    "small_win60_T1": (False, 60, 1, [1]),
    "small_win60_T127": (False, 60, 127, [127, 1, 2, 64]),
    "small_win64_T128": (False, 64, 128, [128, 3, 127]),
    "small_win64_T129": (False, 64, 129, [129, 128, 1]),
    "small_win60_T1000": (False, 60, 1000, [1000, 999, 513, 2]),
    "full_T1": (True, 1200, 1, [1]),
    "full_T129": (True, 1200, 129, [129, 3, 1]),
    "full_T1000": (True, 1200, 1000, [1000, 400]),
}
_models = {}


def _spec_model(full, win, precision, dev):
    key = (full, win)
    if key not in _models:
        _models[key] = _model({"win_size": win}, full=full).to(dev)
    m = _models[key]
    m.precision = precision
    return m


@pytest.mark.parametrize("case", list(SPEC_CASES))
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_spectrogram_against_float64(cuda_device, case, precision):
    full, win, T, lengths = SPEC_CASES[case]
    m = _spec_model(full, win, precision, cuda_device)
    n_fft = 2 * (m.posterior_encoder.in_channels - 1)
    hop = 300 if full else 15
    wav = _wav(T + len(lengths), len(lengths), T * hop)
    got = m.spectrogram(wav.to(cuda_device), torch.tensor(lengths, dtype=torch.int32, device=cuda_device)).cpu().double()
    exact, S = direct_spectrogram(wav, lengths, n_fft=n_fft, hop=hop, win_length=win)
    got = got.numpy()
    Sn = S[:, None, :]
    valid = np.zeros_like(S, dtype=bool)
    for b, n in enumerate(lengths):
        valid[b, :n] = True
        assert np.all(got[b, :, n:] == 0), "frames beyond lengths must be 0"
    r_exact = (np.abs(got - exact) / np.maximum(Sn, 1e-30)).max(axis=1)[valid]
    if precision == "bf16":
        ref, _ = direct_spectrogram(wav, lengths, n_fft=n_fft, hop=hop, win_length=win, bf16=True)
        excess = np.abs(got - ref) - 2.0 ** -8 * np.abs(ref)                 # output rounding to bf16: <= 1 ulp
        r_ops = (np.maximum(excess, 0) / np.maximum(Sn, 1e-30)).max(axis=1)[valid]
        print(f"spectrogram bf16 {case}: vs bf16 operands {r_ops.max():.2e} S, vs exact {r_exact.max():.2e} S")
        assert r_ops.max() <= 5e-8
        assert r_exact.max() <= 2.0 ** -7
    else:
        print(f"spectrogram {precision} {case}: vs exact {r_exact.max():.2e} S")
        assert r_exact.max() <= 2.5e-6
    # first and last valid frame of every utterance on their own (the reflected edges)
    for b, n in enumerate(lengths):
        for f in {0, n - 1}:
            e = np.abs(got[b, :, f] - exact[b, :, f]).max() / S[b, f]
            assert e <= (2.0 ** -7 if precision == "bf16" else 2.5e-6), (b, f, e)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_spectrogram_matches_torch_stft_reference(cuda_device, precision):
    """The stft-based statement (reflect pad per utterance, torch.stft) at the full config, ragged lengths."""
    m = _spec_model(True, 1200, precision, cuda_device)
    lengths = [400, 3, 250]
    wav = _wav(7, 3, 400 * 300)
    got = m.spectrogram(wav.to(cuda_device), torch.tensor(lengths, dtype=torch.int32, device=cuda_device)).cpu().double()
    ref = linear_spectrogram(wav, lengths, n_fft=2048, hop=300, win_length=1200)
    rel = float((got - ref).norm() / ref.norm())
    print(f"spectrogram {precision} vs torch.stft statement: rel-L2 {rel:.2e}")
    assert rel <= (4.5e-3 if precision == "bf16" else 1e-6)


def _convert(m, dev, lengths, T, hop, seed, src, tgt, wav=None, spec=None):
    g = torch.Generator().manual_seed(seed)
    B = len(lengths)
    noise = torch.randn(B, m.hidden_size, T, generator=g).to(dev)
    kw = dict(lengths=torch.tensor(lengths, dtype=torch.int32, device=dev), spk_id=src, tgt_spk_id=tgt, noise=noise)
    if wav is not None:
        return m.voice_conversion(wav=wav.to(dev), **kw), noise
    return m.voice_conversion(spec=spec.to(dev), **kw), noise


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_utterance_alone_equals_inside_ragged_batch(cuda_device, precision):
    m = _spec_model(False, 60, precision, cuda_device)
    T, hop = 200, 15
    wav = _wav(3, 3, T * hop)
    lengths = [200, 77, 1]
    g = torch.Generator().manual_seed(11)
    noise = torch.randn(3, 32, T, generator=g).to(cuda_device)
    ln = torch.tensor(lengths, dtype=torch.int32, device=cuda_device)
    out = m.voice_conversion(wav=wav.to(cuda_device), lengths=ln, spk_id=[0, 1, 1], tgt_spk_id=[1, 0, 0], noise=noise)
    for b, n in enumerate(lengths):
        one = m.voice_conversion(wav=wav[b:b + 1, :n * hop].to(cuda_device), lengths=ln[b:b + 1],
                                 spk_id=[[0, 1, 1][b]], tgt_spk_id=[[1, 0, 0][b]], noise=noise[b:b + 1, :, :n].contiguous())
        assert torch.equal(out["spec"][b, :, :n], one["spec"][0]), b
        assert torch.equal(out["z"][b, :, :n], one["z"][0]), b


def _chain(m, dev, precision, lengths, T, src, tgt, noise, wav=None, spec=None):
    """vsg_spectrogram -> vsg_posterior_forward -> vsg_flow_forward(reverse=0) -> vsg_infer_zp, public calls only."""
    from visinger_b200 import _lib
    L = _lib.lib()
    prec = PREC[precision]
    B, H = len(lengths), m.hidden_size
    ln = torch.tensor(lengths, dtype=torch.int32, device=dev)
    mask = (torch.arange(T, device=dev)[None] < ln[:, None]).float().unsqueeze(1).contiguous()
    if spec is None:
        spec = m.spectrogram(wav.to(dev), ln)
    spec = spec.to(dev).contiguous()
    pe = m.posterior_encoder
    ec = _lib.VsgEncConfig(pe.in_channels, pe.out_channels, pe.hidden_channels, pe.kernel_size, pe.dilation_rate,
                           pe.n_layers, pe.gin_channels)
    ep = _lib.EncPack(ec, dict(m.state_dict()), "posterior_encoder.", dev)
    w = m.spk_id_proj.weight.detach()
    g_src = w[torch.as_tensor(src)].to(dev).unsqueeze(-1).contiguous()
    g_tgt = w[torch.as_tensor(tgt)].to(dev).unsqueeze(-1).contiguous()
    z = torch.empty(B, H, T, device=dev)
    stats = torch.empty(B, 2 * H, T, device=dev)
    st = _lib.stream_ptr(dev)
    ws = torch.empty(ep.workspace_bytes(B, T, prec), dtype=torch.uint8, device=dev)
    _lib.check(L.vsg_posterior_forward(ep.handle, spec.data_ptr(), mask.data_ptr(), g_src.data_ptr(), noise.data_ptr(),
                                       z.data_ptr(), stats.data_ptr(), B, T, prec, ws.data_ptr(), ws.numel(), st), "post")
    hot = m._hot
    hot.precision = precision
    pk = hot._pack()
    ws = torch.empty(pk.workspace_bytes(B, T, prec), dtype=torch.uint8, device=dev)
    z_p = torch.empty_like(z)
    _lib.check(L.vsg_flow_forward(pk.handle, z.data_ptr(), mask.data_ptr(), g_src.data_ptr(), z_p.data_ptr(), B, T, 0, prec,
                                  ws.data_ptr(), ws.numel(), st), "flow")
    wav_out, z_hat = hot.infer_zp(z_p, mask, g_tgt)
    return wav_out.squeeze(1), z_hat, spec


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("source", ["wav", "spec"])
def test_one_call_equals_chain_of_public_calls(cuda_device, precision, source):
    m = _spec_model(False, 60, precision, cuda_device)
    T, hop, lengths = 150, 15, [150, 61]
    wav = _wav(5, 2, T * hop)
    spec_in = None
    if source == "spec":
        spec_in = linear_spectrogram(wav, lengths, n_fft=64, hop=15, win_length=60).float()
    out, noise = _convert(m, cuda_device, lengths, T, hop, 9, [0, 1], [1, 0], wav=wav if source == "wav" else None,
                          spec=spec_in)
    w_ref, z_ref, s_ref = _chain(m, cuda_device, precision, lengths, T, [0, 1], [1, 0], noise,
                                 wav=wav if source == "wav" else None, spec=spec_in)
    assert torch.equal(out["spec"].to(cuda_device), s_ref)
    assert torch.equal(out["z"], z_ref)
    assert torch.equal(out["wav_out"], w_ref)


def _oracle_case(m, lengths, T, hop, win, src, tgt, seed):
    from oracle import visinger_oracle as O
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    n_fft = 2 * (m.posterior_encoder.in_channels - 1)
    wav = _wav(seed, len(lengths), T * hop)
    spec = linear_spectrogram(wav, lengths, n_fft=n_fft, hop=hop, win_length=win).float()
    mask = (torch.arange(T)[None] < torch.tensor(lengths)[:, None]).float().unsqueeze(1)
    w = sd["spk_id_proj.weight"]
    g_src, g_tgt = w[torch.tensor(src)].unsqueeze(-1), w[torch.tensor(tgt)].unsqueeze(-1)
    noise = torch.randn(len(lengths), m.hidden_size, T, generator=torch.Generator().manual_seed(seed + 1))
    hp = m.hparams
    H = m.hidden_size
    post_kw = dict(out_channels=H, hidden=H, kernel_size=5, dilation_rate=1, n_layers=16)
    flow_kw = dict(channels=H, hidden=H, kernel_size=5, dilation_rate=1, n_layers=4, n_flows=4)
    dec_kw = dict(resblock=hp["dec_blocks"], resblock_kernel_sizes=hp["dec_kernel_size"],
                  resblock_dilation_sizes=hp["dec_dilation_sizes"], upsample_rates=hp["upsample_rates"],
                  upsample_kernel_sizes=hp["upsample_kernel_sizes"])
    with torch.no_grad():
        wav_ref, z_ref = voice_conversion(sd, spec, mask, g_src, g_tgt, noise, post_kw=post_kw, flow_kw=flow_kw,
                                          dec_kw=dec_kw)
    return wav, spec, noise, wav_ref, z_ref


ORACLE_GATES = {"fp32": 1.5e-7, "bf16x3": 3e-6, "bf16": 1.3e-2}   # floors in the module docstring


@pytest.mark.parametrize("config", ["small", "full"])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_against_cpu_oracle_composition(cuda_device, config, precision):
    full = config == "full"
    if full:
        m = _model({"num_spk": 4, "win_size": 1200}, full=True, seed=3, precision=precision).to(cuda_device)
        lengths, T, hop, win, src, tgt = [400, 257], 400, 300, 1200, [0, 2], [3, 1]
    else:
        m = _model({"win_size": 60}, seed=3, precision=precision).to(cuda_device)
        lengths, T, hop, win, src, tgt = [300, 170, 9], 300, 15, 60, [0, 1, 0], [1, 0, 1]
    key = (config, "oracle")
    if key not in _models:
        _models[key] = _oracle_case(m.cpu(), lengths, T, hop, win, src, tgt, seed=21)
        m = m.to(cuda_device)
    wav, spec, noise, wav_ref, z_ref = _models[key]
    dev = cuda_device
    out = m.voice_conversion(spec=spec.to(dev), lengths=torch.tensor(lengths, dtype=torch.int32, device=dev), spk_id=src,
                             tgt_spk_id=tgt, noise=noise.to(dev))
    got = out["wav_out"].cpu()
    e_w, e_z = maxabs(got, wav_ref), maxabs(out["z"].cpu(), z_ref)
    rel = float((got - wav_ref).norm() / wav_ref.norm())
    print(f"voice conversion vs oracle {config} {precision}: waveform max-abs {e_w:.3e}, rel-L2 {rel:.3e}, z {e_z:.3e}")
    if precision == "bf16":
        assert rel <= ORACLE_GATES["bf16"]
    else:
        assert e_w <= ORACLE_GATES[precision]
    # from the waveform too: the native spectrogram in place of the float64 one
    out_w = m.voice_conversion(wav=wav.to(dev), lengths=torch.tensor(lengths, dtype=torch.int32, device=dev), spk_id=src,
                               tgt_spk_id=tgt, noise=noise.to(dev))
    rel_w = float((out_w["wav_out"].cpu() - wav_ref).norm() / wav_ref.norm())
    e_ww = maxabs(out_w["wav_out"].cpu(), wav_ref)
    print(f"voice conversion from wav vs oracle {config} {precision}: waveform max-abs {e_ww:.3e}, rel-L2 {rel_w:.3e}")
    if precision == "bf16":
        assert rel_w <= ORACLE_GATES["bf16"]
    else:
        assert e_ww <= ORACLE_GATES[precision]


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
def test_cuda_graph_replay_equals_eager(cuda_device, precision):
    from visinger_b200 import _lib
    m = _spec_model(False, 60, precision, cuda_device)
    dev = cuda_device
    T, B = 120, 2
    pack = m._convert_pack(dev)
    prec = PREC[precision]
    wav = _wav(8, B, T * 15).to(dev)
    ln = torch.tensor([120, 50], dtype=torch.int32, device=dev)
    seeds = torch.tensor([5, 6], dtype=torch.int64, device=dev)
    src, tgt = torch.tensor([0, 1]), torch.tensor([1, 1])
    outs = [torch.empty(B, T * 15, device=dev) for _ in range(2)]
    zs = [torch.empty(B, 32, T, device=dev) for _ in range(2)]
    ws = torch.empty(pack.convert_workspace_bytes(B, T, prec), dtype=torch.uint8, device=dev)
    L = _lib.lib()

    def run(i):
        _lib.check(L.vsg_model_convert(pack.handle, wav.data_ptr(), None, ln.data_ptr(), src.data_ptr(), None,
                                       tgt.data_ptr(), None, None, seeds.data_ptr(), outs[i].data_ptr(), None,
                                       zs[i].data_ptr(), B, T, prec, ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)),
                   "vsg_model_convert")
    s = torch.cuda.Stream(dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        run(0)
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run(1)
    graph.replay()
    torch.cuda.synchronize(dev)
    assert torch.equal(outs[0], outs[1]) and torch.equal(zs[0], zs[1])


def test_model_forward_on_convert_pack_equals_model_pack(cuda_device):
    from visinger_b200 import _lib
    from model_inputs import synth_utterances
    m = _spec_model(False, 60, "bf16", cuda_device)
    dev = cuda_device
    b = synth_utterances(seed=4, n=2, lengths=[90, 60], n_spk=2)
    noise = torch.randn(2, 32, 90, generator=torch.Generator().manual_seed(1)).to(dev)
    args = (b["text_tokens"].to(dev), b["note_pitch"].to(dev), b["note_dur"].to(dev), b["mel2ph"].to(dev))
    ref = m.forward_native(*args, spk_id=b["spk_ids"], noise=noise)["wav_out"].clone()
    conv = m._convert_pack(dev)
    m.__dict__["_native_pack"] = (m.__dict__["_native_pack"][0], conv)   # forward_native through the convert pack
    try:
        got = m.forward_native(*args, spk_id=b["spk_ids"], noise=noise)["wav_out"]
    finally:
        del m.__dict__["_native_pack"]
    assert torch.equal(got, ref)


def test_errors_launch_nothing(cuda_device):
    from visinger_b200 import _lib
    L = _lib.lib()
    dev = cuda_device
    m = _spec_model(False, 60, "bf16", dev)
    conv = m._convert_pack(dev)
    model_only = m._model_pack(dev)
    B, T = 2, 40
    wav = torch.zeros(B, T * 15, device=dev)
    spec = torch.zeros(B, 33, T, device=dev)
    ln = torch.tensor([40, 20], dtype=torch.int32, device=dev)
    seeds = torch.tensor([1, 2], dtype=torch.int64, device=dev)
    out = torch.empty(B, T * 15, device=dev)
    ids, bad = torch.tensor([0, 1]), torch.tensor([0, 2])
    ws = torch.empty(conv.convert_workspace_bytes(B, T, 1), dtype=torch.uint8, device=dev)

    def call(pack=conv, w=wav, s=None, src=ids, tgt=ids, nbytes=None):
        rc = L.vsg_model_convert(pack.handle, w.data_ptr() if w is not None else None, s.data_ptr() if s is not None else None,
                                 ln.data_ptr(), src.data_ptr(), None, tgt.data_ptr(), None, None, seeds.data_ptr(),
                                 out.data_ptr(), None, None, B, T, 1, ws.data_ptr(),
                                 ws.numel() if nbytes is None else nbytes, _lib.stream_ptr(dev))
        return rc, L.vsg_last_launch_count(), L.vsg_last_error()

    assert call()[0] == 0
    for kw, code, word in [(dict(w=None), VSG_EINVAL, b"exactly one"), (dict(s=spec), VSG_EINVAL, b"exactly one"),
                           (dict(pack=model_only), VSG_EINVAL, b"posterior"), (dict(tgt=bad), VSG_EINVAL, b"tgt_spk_id"),
                           (dict(src=bad), VSG_EINVAL, b"src_spk_id"), (dict(nbytes=1024), VSG_ENOMEM, b"workspace")]:
        rc, n, msg = call(**kw)
        assert rc == code and n == 0 and word in msg, (kw, rc, n, msg)
    # pack creation: a bad window and a missing posterior entry (named)
    h = ctypes.c_void_p()
    sd = {k: v.detach().cpu().float().contiguous() for k, v in m.state_dict().items()}
    for drop, win, word in [(None, 65, b"win_length"), ("posterior_encoder.enc.res_skip_layers.7.weight_v", 60,
                                                         b"posterior_encoder.enc.res_skip_layers.7")]:
        host = {k: v for k, v in sd.items() if k != drop}
        arr, keep = _lib._weight_table(host)
        rc = L.vsg_convert_pack_create(ctypes.byref(m._model_config()), arr, len(host), b"", win, dev.index or 0,
                                       ctypes.byref(h))
        assert rc == VSG_EINVAL and word in L.vsg_last_error() and not h.value, (drop, rc, L.vsg_last_error())
