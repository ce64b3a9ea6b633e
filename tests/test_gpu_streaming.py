"""Streaming synthesis on the GPU: vsg_infer_zp_window / vsg_generator_forward_window against the one-pass calls, bit for
bit (torch.equal) in every precision, and the workspace and argument rules of the window calls."""
import ctypes
import random

import pytest
import torch

from helpers import FLOW_FULL, GEN_FULL, gen_cfg_of, load_npz
from streaming_context import dec_context, flow_context

pytestmark = pytest.mark.gpu

PRECISIONS = ["fp32", "bf16", "bf16x3"]
# a small configuration the tensor-core kernels take: stages of 32 and 16 channels at 3 and 9 samples per frame, so the
# row-packed kernels (2 and 4 time steps per row) and conv_post (4 / 2 samples per row) need windows on phase boundaries
FLOW_SMALL = dict(channels=32, hidden=32, kernel_size=5, dilation_rate=1, n_layers=2, n_flows=2, gin=16)
GEN_SMALL = dict(initial_channel=32, resblock="1", rk=[3, 5], rd=[[1, 3], [1, 3]], ur=[3, 3], uic=64, uk=[7, 7], gin=16)
CONFIGS = {"full": (FLOW_FULL, GEN_FULL), "small": (FLOW_SMALL, GEN_SMALL)}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


_hp_cache = {}


def hot_path(name, precision, dev):
    from visinger_b200.models.visinger import HotPath
    key = (name, precision)
    if key not in _hp_cache:
        f, g = CONFIGS[name]
        _hp_cache[key] = HotPath.random_init(f, g, dev, precision=precision, seed=11)
    return _hp_cache[key]


def inputs(name, B, T, lengths, dev, seed=0):
    f, _ = CONFIGS[name]
    gen = torch.Generator().manual_seed(seed)
    z_p = torch.randn(B, f["channels"], T, generator=gen)
    mask = torch.ones(B, 1, T)
    for b, n in enumerate(lengths):
        mask[b, :, n:] = 0
    g = 0.1 * torch.randn(B, f["gin"], 1, generator=gen)
    return (z_p * mask).to(dev), mask.to(dev), g.to(dev)


def L():
    from visinger_b200 import _lib
    return _lib.lib()


def run_window(hp, z_p, mask, g, t0, t1, ws=None, z_q=True):
    """One vsg_infer_zp_window call: (rc, wav [B, (t1 - t0) * hop], z_q [B, C, t1 - t0])."""
    from visinger_b200 import _lib
    B, C, T = z_p.shape
    pack, prec, hop = hp._pack(), _lib.precision_code(hp.precision), hp.decoder.hop_size
    wav = torch.full((B, max(t1 - t0, 0) * hop), float("nan"), device=z_p.device)
    zq = torch.full((B, C, max(t1 - t0, 0)), float("nan"), device=z_p.device) if z_q else None
    if ws is None:
        ws = torch.empty(pack.window_workspace_bytes(B, T, max(t1 - t0, 1), prec), dtype=torch.uint8, device=z_p.device)
    rc = L().vsg_infer_zp_window(pack.handle, z_p.data_ptr(), mask.data_ptr(), g.data_ptr(), wav.data_ptr(),
                                 max(t1 - t0, 0) * hop, zq.data_ptr() if z_q else None, B, T, t0, t1, prec,
                                 ws.data_ptr(), ws.numel(), _lib.stream_ptr(z_p.device))
    return rc, wav, zq


def partitions(T, rng):
    """Chunkings of [0, T): fixed sizes 1, 7, 64, 250, T, and random boundaries (t0 = 0 and t1 = T included)."""
    out = [[(t, min(T, t + n)) for t in range(0, T, n)] for n in (1, 7, 64, 250, T)]
    cuts = sorted(set(rng.sample(range(1, T), min(T - 1, 9))))
    b = [0] + cuts + [T]
    out.append(list(zip(b[:-1], b[1:])))
    return out


@pytest.mark.parametrize("name", ["full", "small"])
def test_window_context_matches_python_formula(dev, name):
    f, g = CONFIGS[name]
    hp = hot_path(name, "fp32", dev)
    assert hp._pack().window_context() == (flow_context(f), dec_context(g))
    if name == "full":
        assert hp._pack().window_context() == (32, 20)


@pytest.mark.parametrize("golden", ["small_gen", "small_gen_rb2"])
def test_window_context_of_golden_decoders(dev, golden):
    from visinger_b200 import _lib
    from visinger_b200.modules.visinger.decoder import Generator
    cfg = gen_cfg_of(load_npz(golden))
    m = Generator(cfg["initial_channel"], cfg["resblock"], cfg["rk"], cfg["rd"], cfg["ur"], cfg["uic"], cfg["uk"],
                  gin_channels=cfg["gin"]).to(dev)
    cf, cd = ctypes.c_int32(), ctypes.c_int32()
    assert L().vsg_window_context(m._pack().handle, ctypes.byref(cf), ctypes.byref(cd)) == 0
    assert (cf.value, cd.value) == (0, dec_context(cfg))


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["full", "small"])
def test_concatenated_windows_equal_one_pass(dev, name, precision):
    hp = hot_path(name, precision, dev)
    B, T = 3, 300
    lengths = [300, 171, 40]   # windows wholly past an utterance's end too
    z_p, mask, g = inputs(name, B, T, lengths, dev, seed=1)
    wav_ref, zq_ref = hp.infer_zp(z_p, mask, g)
    wav_ref = wav_ref.reshape(B, -1)
    hop = hp.decoder.hop_size
    rng = random.Random(7)
    for part in partitions(T, rng):
        wavs, zqs = [], []
        for t0, t1 in part:
            rc, w, zq = run_window(hp, z_p, mask, g, t0, t1)
            assert rc == 0, (t0, t1)
            wavs.append(w)
            zqs.append(zq)
        n = part[1][1] - part[1][0] if len(part) > 1 else T
        assert torch.equal(torch.cat(wavs, 1), wav_ref), (name, precision, n)
        assert torch.equal(torch.cat(zqs, 2), zq_ref), (name, precision, n)
    # out of order, and windows narrower than the context, give the same bits
    part = [(t, min(T, t + 5)) for t in range(0, T, 5)]
    rng.shuffle(part)
    for t0, t1 in part[:20]:
        rc, w, zq = run_window(hp, z_p, mask, g, t0, t1)
        assert rc == 0 and torch.equal(w, wav_ref[:, t0 * hop:t1 * hop]) and torch.equal(zq, zq_ref[:, :, t0:t1])


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["full", "small"])
def test_decoder_windows_equal_one_pass(dev, name, precision):
    hp = hot_path(name, precision, dev)
    B, T = 2, 257
    z, _, g = inputs(name, B, T, [T, T], dev, seed=2)
    ref = hp.decode(z, g)
    hop = hp.decoder.hop_size
    for part in partitions(T, random.Random(3))[1:]:
        got = torch.cat([hp.decode_window(z, g, t0, t1) for t0, t1 in part], 2)
        assert torch.equal(got, ref), (name, precision, part[:2])
    for t0, t1 in ((0, 1), (T - 1, T), (100, 103)):
        assert torch.equal(hp.decode_window(z, g, t0, t1), ref[:, :, t0 * hop:t1 * hop])


@pytest.mark.parametrize("precision", PRECISIONS)
def test_window_in_cuda_graph_replays_same_bits(dev, precision):
    from visinger_b200 import _lib
    hp = hot_path("full", precision, dev)
    B, T, t0, t1 = 2, 400, 130, 230
    z_p, mask, g = inputs("full", B, T, [T, 300], dev, seed=4)
    wav_ref, zq_ref = hp.infer_zp(z_p, mask, g)
    hop = hp.decoder.hop_size
    pack, prec = hp._pack(), _lib.precision_code(precision)
    ws = torch.empty(pack.window_workspace_bytes(B, T, t1 - t0, prec), dtype=torch.uint8, device=dev)
    wav = torch.empty(B, (t1 - t0) * hop, device=dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))

    def call():
        rc = L().vsg_infer_zp_window(pack.handle, z_p.data_ptr(), mask.data_ptr(), g.data_ptr(), wav.data_ptr(),
                                     (t1 - t0) * hop, None, B, T, t0, t1, prec, ws.data_ptr(), ws.numel(),
                                     _lib.stream_ptr(dev))
        assert rc == 0

    with torch.cuda.stream(side):
        call()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call()
    wav.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize(dev)
    assert torch.equal(wav, wav_ref.reshape(B, -1)[:, t0 * hop:t1 * hop])


def test_workspace_does_not_grow_with_T_and_is_exact(dev):
    from visinger_b200 import _lib
    for prec in PRECISIONS:
        hp = hot_path("full", prec, dev)
        pack, code = hp._pack(), _lib.precision_code(prec)
        sizes = [pack.window_workspace_bytes(4, T, 250, code) for T in (1000, 4600, 14400, 100000)]
        assert all(s > 0 for s in sizes) and max(sizes) == sizes[0], (prec, sizes)
        assert sizes[0] < pack.workspace_bytes(4, 1000, code)
    hp = hot_path("full", "bf16", dev)
    B, T = 2, 500
    z_p, mask, g = inputs("full", B, T, [T, 321], dev, seed=5)
    wav_ref, _ = hp.infer_zp(z_p, mask, g)
    hop, code = hp.decoder.hop_size, _lib.precision_code("bf16")
    n = hp._pack().window_workspace_bytes(B, T, 64, code)
    ws = torch.empty(n, dtype=torch.uint8, device=dev)
    for t0 in (0, 200, T - 64):   # clipped at either end and interior: all fit in exactly that many bytes
        rc, w, _ = run_window(hp, z_p, mask, g, t0, t0 + 64, ws=ws, z_q=False)
        assert rc == 0 and torch.equal(w, wav_ref.reshape(B, -1)[:, t0 * hop:(t0 + 64) * hop])
    rc, w, _ = run_window(hp, z_p, mask, g, 200, 264, ws=ws[:n - 1], z_q=False)
    assert rc == -3 and _lib.last_launch_count() == 0


def test_window_argument_errors_before_any_launch(dev):
    from visinger_b200 import _lib
    hp = hot_path("full", "bf16", dev)
    B, T = 2, 100
    z_p, mask, g = inputs("full", B, T, [T, T], dev)
    pack, code, hop = hp._pack(), _lib.precision_code("bf16"), hp.decoder.hop_size
    ws = torch.empty(pack.window_workspace_bytes(B, T, T, code), dtype=torch.uint8, device=dev)
    wav = torch.empty(B, T * hop, device=dev)
    s = _lib.stream_ptr(dev)

    def call(t0=10, t1=20, wav_ld=10 * hop, zp=z_p.data_ptr(), m=mask.data_ptr(), w=wav.data_ptr(), nbytes=ws.numel()):
        return L().vsg_infer_zp_window(pack.handle, zp, m, g.data_ptr(), w, wav_ld, None, B, T, t0, t1, code,
                                       ws.data_ptr(), nbytes, s)

    for kw in (dict(t0=-1), dict(t1=T + 1), dict(t0=20, t1=20), dict(t0=30, t1=20), dict(zp=None), dict(m=None),
               dict(w=None), dict(wav_ld=10 * hop - 1)):
        assert call(**kw) == -1, kw
        assert _lib.last_launch_count() == 0
    assert call(nbytes=100) == -3 and _lib.last_launch_count() == 0
    assert call() == 0 and _lib.last_launch_count() > 0
    rc = L().vsg_generator_forward_window(pack.handle, z_p.data_ptr(), g.data_ptr(), wav.data_ptr(), hop, B, T, 5, 7,
                                          code, ws.data_ptr(), ws.numel(), s)
    assert rc == -1 and _lib.last_launch_count() == 0


@pytest.mark.parametrize("precision", PRECISIONS)
def test_forward_streaming_equals_infer_zp_small_model(dev, precision):
    from model_inputs import SMALL_HPARAMS, synth_utterances
    from visinger_b200.models.visinger import VISinger
    torch.manual_seed(2)
    m = VISinger(73, 117, 132, SMALL_HPARAMS, precision=precision).eval().to(dev)
    b = synth_utterances(9, 2, min_frames=150, max_frames=400, n_spk=2)
    args = [b[k].to(dev) for k in ("text_tokens", "note_pitch", "note_dur", "mel2ph")]
    B, T = b["mel2ph"].shape
    noise = torch.randn(B, 32, T, generator=torch.Generator().manual_seed(1)).to(dev)
    spk = b["spk_ids"].to(dev)
    z_p, mask, spk_emb = m.prior(*args, spk_id=spk, noise=noise, sample=True)
    m._hot.precision = precision
    ref, _ = m._hot.infer_zp(z_p, mask, spk_emb)
    got = torch.cat(list(m.forward_streaming(*args, spk_id=spk, chunk_frames=37, noise=noise)), 2)
    assert torch.equal(got, ref)


def test_forward_streaming_4600_frames_bf16(dev):
    from model_inputs import full_model_mirror, synth_utterances
    m = full_model_mirror(precision="bf16").to(dev)
    b = synth_utterances(5, 1, lengths=[4600])
    args = [b[k].to(dev) for k in ("text_tokens", "note_pitch", "note_dur", "mel2ph")]
    T = b["mel2ph"].shape[1]
    noise = torch.randn(1, 192, T, generator=torch.Generator().manual_seed(3)).to(dev)
    spk = b["spk_ids"].to(dev)
    z_p, mask, spk_emb = m.prior(*args, spk_id=spk, noise=noise, sample=True)
    m._hot.precision = "bf16"
    ref, _ = m._hot.infer_zp(z_p, mask, spk_emb)
    chunks = list(m.forward_streaming(*args, spk_id=spk, chunk_frames=500, noise=noise))
    assert [c.shape[2] for c in chunks] == [500 * 300] * 9 + [100 * 300]
    assert torch.equal(torch.cat(chunks, 2), ref)
