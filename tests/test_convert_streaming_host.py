"""Streaming voice conversion on the float64 composition of tests/vc_reference.py (spectrogram, posterior, flow both ways,
decoder) at the small config, on the CPU: the window ranges and input span vsg_convert_window_context /
vsg_convert_window_input derive, restated in Python and checked against the composition.

- Dependency traces: the posterior reaches exactly Cp frames each way, and one spectrogram frame reaches no further than
  Cp + 2 Cf + Cd output frames (the flow pair reaches less than 2 Cf: see test_dependency_trace_within_the_context).
- A window computed from a wav that holds NaN outside the window's input span [s0, s1) equals the one pass to 1e-10 (the
  CPU convolutions sum in a length-dependent order), at both utterance ends and for ragged lengths.  That the decoder's and
  the flow's contexts are each needed in full is tests/test_streaming_host.py's finding."""
import math

import pytest
import torch

from model_inputs import SMALL_HPARAMS
from oracle import visinger_oracle as O
from streaming_context import dec_context, flow_context
from vc_reference import linear_spectrogram

WIN = 60
HP = dict(SMALL_HPARAMS, win_size=WIN)
HOP = 15
N_FFT = 2 * (HP["num_linear_bins"] - 1)
POST_CFG = dict(kernel_size=5, dilation_rate=1, n_layers=16, n_flows=1)     # PosteriorEncoder(..., 5, 1, 16, gin)
FLOW_CFG = dict(kernel_size=5, dilation_rate=1, n_layers=4, n_flows=4)
GEN_CFG = dict(resblock=HP["dec_blocks"], rk=HP["dec_kernel_size"], rd=HP["dec_dilation_sizes"], ur=HP["upsample_rates"],
               uk=HP["upsample_kernel_sizes"])
CP, CF, CD = flow_context(POST_CFG), flow_context(FLOW_CFG), dec_context(GEN_CFG)
CTX = CP + 2 * CF + CD


def test_small_config_context():
    assert (CP, CF, CD) == (32, 32, CD) and CD > 0


def ranges(T, t0, t1):
    """window_ranges at fp32 (no alignment, no minimum length): decoder, flow reverse, flow forward, posterior."""
    da, db = max(0, t0 - CD), min(T, t1 + CD)
    grow = lambda c: (max(0, da - c), min(T, db + c))   # noqa: E731
    return (da, db), grow(CF), grow(2 * CF), grow(2 * CF + CP)


def input_span(T, t0, t1):
    """vsg_convert_window_input: rows pa .. pb + taps - 2 of hop samples from sample q * hop + off, and every sample
    below pb * hop (the masks of the posterior's frames)."""
    _, _, _, (pa, pb) = ranges(T, t0, t1)
    off = (N_FFT - WIN) // 2 - (N_FFT - HOP) // 2
    taps = math.ceil(WIN / HOP)
    return max(0, pa * HOP + off), min(T * HOP, max(pb * HOP, (pb + taps - 1) * HOP + off))


_case = {}


def setup():
    if not _case:
        from visinger_b200.models.visinger import VISinger
        torch.manual_seed(3)
        m = VISinger(73, 117, 132, HP).eval()
        sd = {k: v.detach().double() for k, v in m.state_dict().items()}
        gen = torch.Generator().manual_seed(5)
        for f in range(4):   # the reference zero-initialises the flow's `post`: give the couplings something to do
            for k in ("weight", "bias"):
                key = f"flow.flows.{2 * f}.post.{k}"
                sd[key] = 0.05 * torch.randn(sd[key].shape, generator=gen, dtype=torch.float64)
        w = sd["spk_id_proj.weight"]
        _case.update(sd=sd, g_src=w[[0, 1]].unsqueeze(-1), g_tgt=w[[1, 0]].unsqueeze(-1))
    return _case


def _wav(seed, B, L):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(L, dtype=torch.float64)
    f = 0.01 + 0.2 * torch.rand(B, 1, generator=g, dtype=torch.float64)
    return 0.5 * torch.sin(f * t) + 0.1 * torch.randn(B, L, generator=g, dtype=torch.float64)


def _mask(lengths, T):
    return (torch.arange(T)[None] < torch.tensor(lengths)[:, None]).double().unsqueeze(1)


def compose(spec, mask, noise, a=None):
    """The composition over frames [0, T) of its inputs; `a` = ranges(...) runs each part over its own range only and
    returns the decoder's range [da, db)."""
    c = setup()
    sd, H = c["sd"], HP["hidden_size"]
    T = spec.shape[2]
    (da, db), (fa, fb), (ga, gb), (pa, pb) = a or ((0, T),) * 4
    post_kw = dict(out_channels=H, hidden=H, kernel_size=5, dilation_rate=1, n_layers=16)
    flow_kw = dict(channels=H, hidden=H, kernel_size=5, dilation_rate=1, n_layers=4, n_flows=4)
    dec_kw = dict(resblock=HP["dec_blocks"], resblock_kernel_sizes=HP["dec_kernel_size"],
                  resblock_dilation_sizes=HP["dec_dilation_sizes"], upsample_rates=HP["upsample_rates"],
                  upsample_kernel_sizes=HP["upsample_kernel_sizes"])
    B = spec.shape[0]
    g_src, g_tgt = c["g_src"][:B], c["g_tgt"][:B]
    z, _, _ = O.posterior_encoder(sd, spec[:, :, pa:pb], mask[:, :, pa:pb], g_src, noise[:, :, pa:pb],
                                  prefix="posterior_encoder.", **post_kw)
    z_p = O.flow(sd, z[:, :, ga - pa:gb - pa], mask[:, :, ga:gb], g=g_src, reverse=False, prefix="flow.", **flow_kw)
    z_hat = O.flow(sd, z_p[:, :, fa - ga:fb - ga], mask[:, :, fa:fb], g=g_tgt, reverse=True, prefix="flow.",
                   **flow_kw) * mask[:, :, fa:fb]
    x = z_hat[:, :, da - fa:db - fa] * mask[:, :, da:db]
    return O.generator(sd, x, g=g_tgt, prefix="decoder.", **dec_kw).squeeze(1)


def _trace(fn, x, F):
    """(left, right): how far the frames that perturbing input frame F changes reach."""
    y0 = fn(x)
    x1 = x.clone()
    x1[:, :, F] += 1.0
    changed = ((fn(x1) - y0).abs().amax(dim=tuple(range(y0.dim() - 1))) > 0).nonzero().flatten()
    return int(F - changed.min()), int(changed.max() - F)


def test_dependency_trace_within_the_context():
    """Each part's reach is its own context (posterior Cp, decoder Cd: both tight), and the whole chain's stays within
    Cp + 2 Cf + Cd.  The flow pair reaches 2 Cf - Cf / n_flows, not 2 Cf: the forward flow's last coupling and the
    reverse flow's first update the same half from the same, unchanged conditioning half.  The window keeps the plain
    sum of the parts' contexts (each part runs over its own range with its own context), which is the safe bound."""
    c = setup()
    sd, H, T, F = c["sd"], HP["hidden_size"], 2 * CTX + 9, CTX + 4
    mask = _mask([T], T)
    gen = torch.Generator().manual_seed(2)
    noise = torch.randn(1, H, T, generator=gen, dtype=torch.float64)
    spec = torch.rand(1, HP["num_linear_bins"], T, generator=gen, dtype=torch.float64)
    post = lambda s: O.posterior_encoder(sd, s, mask, c["g_src"][:1], noise, prefix="posterior_encoder.",  # noqa: E731
                                         out_channels=H, hidden=H, kernel_size=5, dilation_rate=1, n_layers=16)[0]
    assert _trace(post, spec, F) == (CP, CP)
    kw = dict(channels=H, hidden=H, kernel_size=5, dilation_rate=1, n_layers=4, n_flows=4, prefix="flow.")
    pair = lambda z: O.flow(sd, O.flow(sd, z, mask, g=c["g_src"][:1], **kw), mask, g=c["g_tgt"][:1],  # noqa: E731
                                   reverse=True, **kw)
    z = torch.randn(1, H, T, generator=gen, dtype=torch.float64)
    assert max(_trace(pair, z, F)) == 2 * CF - CF // FLOW_CFG["n_flows"]
    whole = lambda s: compose(s, mask, noise)   # noqa: E731
    wav = _wav(1, 1, T * HOP)
    spec = linear_spectrogram(wav, [T], n_fft=N_FFT, hop=HOP, win_length=WIN)
    y0 = whole(spec)
    spec1 = spec.clone()
    spec1[:, :, F] += 1.0
    changed = ((whole(spec1) - y0).abs()[0] > 0).nonzero().flatten() // HOP
    left, right = int(F - changed.min()), int(changed.max() - F)
    assert CP + 2 * CF <= min(left, right) and max(left, right) <= CTX, (left, right, CTX)


@pytest.mark.parametrize("where", ["interior", "start", "end", "ragged"])
def test_window_from_its_input_span_equals_one_pass(where):
    T = 2 * CTX + 40
    lengths = {"ragged": [T - 30, CTX + 50]}.get(where, [T, T])
    t0, t1 = {"interior": (CTX + 5, CTX + 12), "start": (0, 6), "end": (T - 6, T),
              "ragged": (CTX + 40, CTX + 60)}[where]
    B = len(lengths)
    wav = _wav(3, B, T * HOP)
    mask = _mask(lengths, T)
    noise = torch.randn(B, HP["hidden_size"], T, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    full = compose(linear_spectrogram(wav, lengths, n_fft=N_FFT, hop=HOP, win_length=WIN), mask, noise)
    s0, s1 = input_span(T, t0, t1)
    cut = torch.full_like(wav, float("nan"))
    cut[:, s0:s1] = wav[:, s0:s1]
    a = ranges(T, t0, t1)
    # (frames outside the posterior's range read NaN; compose reads only that range)
    spec = linear_spectrogram(cut, lengths, n_fft=N_FFT, hop=HOP, win_length=WIN)
    da = a[0][0]
    win = compose(spec, mask, noise, a)[:, (t0 - da) * HOP:(t1 - da) * HOP]
    assert torch.isfinite(win).all()
    assert float((win - full[:, t0 * HOP:t1 * HOP]).abs().max()) < 1e-10
