"""Streaming voice conversion on the GPU: vsg_model_convert_window against the one-pass vsg_model_convert, bit for bit
(torch.equal) in every precision, the input span of vsg_convert_window_input, and the workspace and argument rules of
the window call."""
import math
import random

import pytest
import torch

from model_inputs import SMALL_HPARAMS, full_hparams
from streaming_context import dec_context, flow_context

pytestmark = pytest.mark.gpu

VSG_EINVAL, VSG_ENOMEM = -1, -3
PREC = {"fp32": 0, "bf16": 1, "bf16x3": 2}
CONFIGS = {"small": (False, 60, 15), "full": (True, 1200, 300)}   # (full hparams, win_size, hop)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


_models = {}


def model(name, precision, dev):
    from visinger_b200.models.visinger import VISinger
    if name not in _models:
        full, win, _ = CONFIGS[name]
        hp = full_hparams() if full else dict(SMALL_HPARAMS)
        hp.update(win_size=win, num_spk=2)
        torch.manual_seed(1)
        m = VISinger(73, 117, 132, hp).eval()
        with torch.no_grad():   # the reference zero-initialises the flow's `post` (an identity flow): give it weights
            for f in range(4):
                m.flow.flows[2 * f].post.weight.normal_(0, 0.05)
                m.flow.flows[2 * f].post.bias.normal_(0, 0.05)
        _models[name] = m.to(dev)
    m = _models[name]
    m.precision = precision
    return m


def wav_of(seed, B, L, dev):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(L, dtype=torch.float64)
    f = 0.005 + 0.3 * torch.rand(B, 1, generator=g, dtype=torch.float64)
    return (0.4 * torch.sin(f * t) + 0.05 * torch.randn(B, L, generator=g, dtype=torch.float64)).float().to(dev)


class Case:
    """One batch: wav, lengths, speakers, seeds (or noise), and the one pass's wav_out / z_hat."""

    def __init__(self, m, dev, lengths, T, seed, noise=False):
        self.m, self.dev, self.B, self.T = m, dev, len(lengths), T
        self.pack = m._convert_pack(dev)
        self.hop, self.prec = self.pack.hop, PREC[m.precision]
        self.wav = wav_of(seed, self.B, T * self.hop, dev)
        self.ln = torch.tensor(lengths, dtype=torch.int32, device=dev)
        self.src = torch.tensor([b % 2 for b in range(self.B)], dtype=torch.int64)
        self.tgt = 1 - self.src
        g = torch.Generator().manual_seed(seed + 1)
        self.seeds = torch.randint(0, 2 ** 62, (self.B,), generator=g, dtype=torch.int64).to(dev)
        self.noise = torch.randn(self.B, m.hidden_size, T, generator=g).to(dev) if noise else None
        kw = dict(noise=self.noise) if noise else dict(seeds=self.seeds)
        out = m.voice_conversion(wav=self.wav, lengths=self.ln, spk_id=self.src, tgt_spk_id=self.tgt, **kw)
        self.ref_wav, self.ref_z = out["wav_out"], out["z"]

    def ws_bytes(self, n, T=None):
        return self.pack.convert_window_workspace_bytes(self.B, T or self.T, n, self.prec)

    def call(self, t0, t1, ws=None, wav=None, ln=None, wav_ld=None, z=True, nbytes=None, pack=None):
        """(rc, wav_out [B, (t1 - t0) * hop], z_out [B, H, t1 - t0]) of one vsg_model_convert_window call."""
        from visinger_b200 import _lib
        n = max(t1 - t0, 0)
        out = torch.full((self.B, n * self.hop), float("nan"), device=self.dev)
        zo = torch.full((self.B, self.m.hidden_size, n), float("nan"), device=self.dev) if z else None
        if ws is None:
            ws = torch.empty(self.ws_bytes(max(n, 1)), dtype=torch.uint8, device=self.dev)
        w = self.wav if wav is None else wav
        rc = _lib.lib().vsg_model_convert_window(
            (pack or self.pack).handle, w.data_ptr(), (self.ln if ln is None else ln).data_ptr(), self.src.data_ptr(), None,
            self.tgt.data_ptr(), None, self.noise.data_ptr() if self.noise is not None else None,
            None if self.noise is not None else self.seeds.data_ptr(), out.data_ptr(),
            n * self.hop if wav_ld is None else wav_ld, zo.data_ptr() if z else None, self.B, self.T, t0, t1, self.prec,
            ws.data_ptr(), ws.numel() if nbytes is None else nbytes, _lib.stream_ptr(self.dev))
        return rc, out, zo

    def check(self, t0, t1, out, zo):
        assert torch.equal(out, self.ref_wav[:, t0 * self.hop:t1 * self.hop]), (t0, t1)
        assert torch.equal(zo, self.ref_z[:, :, t0:t1]), (t0, t1)


@pytest.mark.parametrize("name", ["small", "full"])
def test_window_context_matches_python_formula(dev, name):
    m = model(name, "fp32", dev)
    hp = m.hparams
    post = dict(kernel_size=5, dilation_rate=1, n_layers=16, n_flows=1)
    flow = dict(kernel_size=5, dilation_rate=1, n_layers=4, n_flows=4)
    gen = dict(resblock=hp["dec_blocks"], rk=hp["dec_kernel_size"], rd=hp["dec_dilation_sizes"], ur=hp["upsample_rates"],
               uk=hp["upsample_kernel_sizes"])
    got = m._convert_pack(dev).convert_window_context()
    assert got == (flow_context(post), flow_context(flow), dec_context(gen))
    if name == "full":
        assert got == (32, 32, 20)


CASES = {   # name: (config, T, lengths): ragged, a one-frame utterance, T shorter than the context
    "small_T200": ("small", 200, [200, 77, 1]),
    "small_T40": ("small", 40, [40, 13]),
    "full_T150": ("full", 150, [150, 61, 1]),
}


@pytest.mark.parametrize("precision", ["fp32", "bf16", "bf16x3"])
@pytest.mark.parametrize("case", list(CASES))
def test_concatenated_windows_equal_one_pass(dev, case, precision):
    name, T, lengths = CASES[case]
    rng = random.Random(3)
    for noise in (False, True):
        c = Case(model(name, precision, dev), dev, lengths, T, seed=T, noise=noise)
        for n in ((1, 7, 64, T) if not noise else (7,)):
            part = [(t, min(T, t + n)) for t in range(0, T, n)]
            order = list(range(len(part)))
            rng.shuffle(order)
            outs, zs = [None] * len(part), [None] * len(part)
            for i in order:
                rc, outs[i], zs[i] = c.call(*part[i])
                assert rc == 0, part[i]
            assert torch.equal(torch.cat(outs, 1), c.ref_wav), (case, precision, n, noise)
            assert torch.equal(torch.cat(zs, 2), c.ref_z), (case, precision, n, noise)


@pytest.mark.parametrize("precision", ["fp32", "bf16", "bf16x3"])
def test_window_reads_only_its_input_span(dev, precision):
    """NaN outside [s0, s1) gives the same bits, and so does any lengths[b] >= ceil(s1 / hop) for an utterance that
    long: a live caller can emit [t0, t1) once samples [0, s1) have arrived."""
    T = 400
    c = Case(model("small", precision, dev), dev, [T, 300, 1], T, seed=9)
    for t0, t1 in ((0, 20), (150, 157), (230, 300), (T - 9, T)):
        s0, s1 = c.pack.convert_window_input(c.B, T, t0, t1, c.prec)
        assert 0 <= s0 < s1 <= T * c.hop and s1 >= t1 * c.hop
        cut = torch.full_like(c.wav, float("nan"))
        cut[:, s0:s1] = c.wav[:, s0:s1]
        rc, out, zo = c.call(t0, t1, wav=cut)
        assert rc == 0
        c.check(t0, t1, out, zo)
        k = math.ceil(s1 / c.hop)
        ln = c.ln.clone()
        for b in range(c.B):
            if int(c.ln[b]) >= k:
                ln[b] = k if b % 2 == 0 else T + 5   # (clamped to T)
        rc, out, zo = c.call(t0, t1, wav=cut, ln=ln)
        assert rc == 0
        c.check(t0, t1, out, zo)


def test_workspace_does_not_grow_with_T_and_is_exact(dev):
    for prec in ("fp32", "bf16", "bf16x3"):
        m = model("full", prec, dev)
        pack, code = m._convert_pack(dev), PREC[prec]
        sizes = [pack.convert_window_workspace_bytes(2, T, 250, code) for T in (1000, 4600, 14400, 100000)]
        assert all(s > 0 for s in sizes) and max(sizes) == sizes[0], (prec, sizes)
        assert sizes[0] < pack.convert_workspace_bytes(2, 1000, code)
    c = Case(model("full", "bf16", dev), dev, [300, 211], 300, seed=4)
    n = c.ws_bytes(64)
    ws = torch.empty(n, dtype=torch.uint8, device=dev)
    for t0 in (0, 120, 300 - 64):   # clipped at either end and interior: all fit in exactly that many bytes
        rc, out, zo = c.call(t0, t0 + 64, ws=ws)
        assert rc == 0
        c.check(t0, t0 + 64, out, zo)
    from visinger_b200 import _lib
    rc, _, _ = c.call(120, 184, ws=ws, nbytes=n - 1)
    assert rc == VSG_ENOMEM and _lib.last_launch_count() == 0


def test_window_argument_errors_before_any_launch(dev):
    from visinger_b200 import _lib
    m = model("small", "bf16", dev)
    c = Case(m, dev, [60, 60], 60, seed=2)
    ws = torch.empty(c.ws_bytes(60), dtype=torch.uint8, device=dev)
    for kw in (dict(t0=-1, t1=5), dict(t0=0, t1=61), dict(t0=20, t1=20), dict(t0=30, t1=20),
               dict(t0=10, t1=20, wav_ld=10 * c.hop - 1), dict(t0=10, t1=20, pack=m._model_pack(dev))):
        t0, t1 = kw.pop("t0"), kw.pop("t1")
        rc, _, _ = c.call(t0, t1, ws=ws, **kw)
        assert rc == VSG_EINVAL and _lib.last_launch_count() == 0, (t0, t1, kw)
    rc, _, _ = c.call(10, 20, ws=ws, nbytes=100)
    assert rc == VSG_ENOMEM and _lib.last_launch_count() == 0
    rc, out, zo = c.call(10, 20, ws=ws)
    assert rc == 0 and _lib.last_launch_count() > 0
    c.check(10, 20, out, zo)


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
def test_window_in_cuda_graph_replays_on_new_wav(dev, precision):
    from visinger_b200 import _lib
    m = model("full", precision, dev)
    B, T, t0, t1 = 2, 300, 100, 180
    c = Case(m, dev, [T, 250], T, seed=5)
    ws = torch.empty(c.ws_bytes(t1 - t0), dtype=torch.uint8, device=dev)
    wav = c.wav.clone()
    out = torch.empty(B, (t1 - t0) * c.hop, device=dev)

    def call():
        rc = _lib.lib().vsg_model_convert_window(
            c.pack.handle, wav.data_ptr(), c.ln.data_ptr(), c.src.data_ptr(), None, c.tgt.data_ptr(), None, None,
            c.seeds.data_ptr(), out.data_ptr(), (t1 - t0) * c.hop, None, B, T, t0, t1, c.prec, ws.data_ptr(), ws.numel(),
            _lib.stream_ptr(dev))
        assert rc == 0

    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        call()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call()
    wav.copy_(wav_of(77, B, T * c.hop, dev))
    out.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize(dev)
    rc, eager, _ = c.call(t0, t1, wav=wav, z=False)
    assert rc == 0 and torch.equal(out, eager)
    assert not torch.equal(out, c.ref_wav[:, t0 * c.hop:t1 * c.hop])   # the replay read the new contents


@pytest.mark.parametrize("precision", ["fp32", "bf16", "bf16x3"])
def test_voice_conversion_streaming_equals_voice_conversion(dev, precision):
    m = model("small", precision, dev)
    T = 230
    wav = wav_of(12, 2, T * 15, dev)
    ln = torch.tensor([T, 150], dtype=torch.int32, device=dev)
    seeds = torch.tensor([3, 4], dtype=torch.int64, device=dev)
    noise = torch.randn(2, 32, T, generator=torch.Generator().manual_seed(8)).to(dev)
    for kw in (dict(seeds=seeds), dict(noise=noise)):
        ref = m.voice_conversion(wav=wav, lengths=ln, spk_id=[0, 1], tgt_spk_id=[1, 0], **kw)["wav_out"]
        chunks = list(m.voice_conversion_streaming(wav, ln, spk_id=[0, 1], tgt_spk_id=[1, 0], chunk_frames=37, **kw))
        assert [ch.shape[1] for ch in chunks] == [37 * 15] * 6 + [8 * 15]
        assert torch.equal(torch.cat(chunks, 1), ref)
    with pytest.raises(RuntimeError, match="lengths"):
        next(m.voice_conversion_streaming(wav, ln[:1], spk_id=[0, 1], tgt_spk_id=[1, 0], seeds=seeds))
