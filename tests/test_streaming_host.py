"""Streaming windows on the CPU oracle: the context formula of tests/streaming_context.py (what vsg_window_context
derives from a pack's config) against a dependency trace, and the oracle windowed with exactly that context against its
own one pass in float64 (to 1e-10: the CPU convolutions sum in a length-dependent order, ~1e-13 apart)."""
import pytest
import torch

from oracle import visinger_oracle as O
from helpers import FLOW_FULL, GEN_FULL, flow_oracle_kw, flow_shapes, gen_oracle_kw, gen_shapes
from streaming_context import dec_context, flow_context

FLOWS = {
    "small": dict(channels=8, hidden=16, kernel_size=5, dilation_rate=1, n_layers=2, n_flows=4, gin=8),
    "dil_odd": dict(channels=4, hidden=8, kernel_size=3, dilation_rate=2, n_layers=3, n_flows=3, gin=0),
}
GENS = {
    "small": dict(initial_channel=8, resblock="1", rk=[3, 7, 11], rd=[[1, 3, 5]] * 3, ur=[5, 3, 2], uic=32, uk=[11, 7, 4],
                  gin=8),
    "rb2": dict(initial_channel=8, resblock="2", rk=[3, 5], rd=[[1, 3], [1, 3]], ur=[4, 2], uic=16, uk=[8, 4], gin=0),
    "odd_rates": dict(initial_channel=8, resblock="1", rk=[3, 5], rd=[[1, 3], [1, 3]], ur=[3, 3], uic=16, uk=[7, 7], gin=0),
}


def test_shipped_config_context():
    assert flow_context(FLOW_FULL) == 32
    assert dec_context(GEN_FULL) == 20


def _flow_setup(cfg, T, seed=3):
    sd = {k: v.double() for k, v in O.synth_state_dict(flow_shapes(cfg), seed).items()}
    for k in sd:
        if ".post." in k:   # the reference zero-initialises post: give the couplings something to do
            sd[k] = 0.05 * torch.randn(sd[k].shape, generator=torch.Generator().manual_seed(7), dtype=torch.float64)
    gen = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(2, cfg["channels"], T, generator=gen, dtype=torch.float64)
    g = 0.1 * torch.randn(2, cfg["gin"], 1, generator=gen, dtype=torch.float64) if cfg["gin"] else None
    return sd, x, g


def _flow(cfg, sd, x, g):
    mask = torch.ones(x.shape[0], 1, x.shape[2], dtype=torch.float64)
    return O.flow(sd, x, mask, g, reverse=True, **flow_oracle_kw(cfg)) * mask


def _gen_setup(cfg, T, seed=5):
    sd = {k: v.double() for k, v in O.synth_state_dict(gen_shapes(cfg), seed).items()}
    gen = torch.Generator().manual_seed(seed + 1)
    z = torch.randn(2, cfg["initial_channel"], T, generator=gen, dtype=torch.float64)
    g = 0.1 * torch.randn(2, cfg["gin"], 1, generator=gen, dtype=torch.float64) if cfg["gin"] else None
    return sd, z, g


def _gen(cfg, sd, z, g):
    return O.generator(sd, z, g, **gen_oracle_kw(cfg)).reshape(z.shape[0], -1)


def _hop(cfg):
    h = 1
    for r in cfg["ur"]:
        h *= r
    return h


@pytest.mark.parametrize("name", sorted(FLOWS))
def test_flow_context_matches_dependency_trace(name):
    cfg = FLOWS[name]
    C = flow_context(cfg)
    T, F = 4 * C + 8, 2 * C + 3
    sd, x, g = _flow_setup(cfg, T)
    y0 = _flow(cfg, sd, x, g)
    x1 = x.clone()
    x1[:, :, F] += 1.0
    changed = ((_flow(cfg, sd, x1, g) - y0).abs().amax(dim=(0, 1)) > 0).nonzero().flatten()
    assert int(F - changed.min()) == C and int(changed.max() - F) == C


@pytest.mark.parametrize("name", sorted(GENS))
def test_decoder_context_matches_dependency_trace(name):
    cfg = GENS[name]
    C, hop = dec_context(cfg), _hop(cfg)
    T, F = 4 * C + 8, 2 * C + 3
    sd, z, g = _gen_setup(cfg, T)
    w0 = _gen(cfg, sd, z, g)
    z1 = z.clone()
    z1[:, :, F] += 1.0
    changed = ((_gen(cfg, sd, z1, g) - w0).abs().amax(dim=0) > 0).nonzero().flatten() // hop
    assert max(int(F - changed.min()), int(changed.max() - F)) == C


@pytest.mark.parametrize("name", sorted(FLOWS))
def test_windowed_flow_oracle(name):
    cfg = FLOWS[name]
    C = flow_context(cfg)
    T, t0, t1 = 4 * C + 10, 2 * C, 2 * C + 7
    sd, x, g = _flow_setup(cfg, T)
    full = _flow(cfg, sd, x, g)[:, :, t0:t1]
    a, b = t0 - C, t1 + C
    win = _flow(cfg, sd, x[:, :, a:b], g)[:, :, t0 - a:t1 - a]
    assert float((win - full).abs().max()) < 1e-10
    # one frame less on a side: the one pass reads a frame that window would not see (the comparison is between two
    # runs of the same length, so any difference is a dependence, not summation order)
    for f in (t0 - C, t1 - 1 + C):
        x1 = x.clone()
        x1[:, :, f] += 1.0
        assert not torch.equal(_flow(cfg, sd, x1, g)[:, :, t0:t1], full), f
    # clipped at the utterance's ends, where the window's zero padding is the utterance's own
    win = _flow(cfg, sd, x[:, :, :C + 5], g)[:, :, :5]
    assert float((win - _flow(cfg, sd, x, g)[:, :, :5]).abs().max()) < 1e-10


@pytest.mark.parametrize("name", sorted(GENS))
def test_windowed_decoder_oracle(name):
    cfg = GENS[name]
    C, hop = dec_context(cfg), _hop(cfg)
    T, t0, t1 = 4 * C + 10, 2 * C, 2 * C + 7
    sd, z, g = _gen_setup(cfg, T)
    w_full = _gen(cfg, sd, z, g)
    full = w_full[:, t0 * hop:t1 * hop]
    a, b = t0 - C, t1 + C
    win = _gen(cfg, sd, z[:, :, a:b], g)[:, (t0 - a) * hop:(t1 - a) * hop]
    assert float((win - full).abs().max()) < 1e-10
    # one frame less on either side that sets C misses a frame the one pass reads (C is the larger of the two reaches)
    for f in (t0 - C, t1 - 1 + C):
        z1 = z.clone()
        z1[:, :, f] += 1.0
        if not torch.equal(_gen(cfg, sd, z1, g)[:, t0 * hop:t1 * hop], full):
            break
    else:
        pytest.fail("no input frame C frames from the window changes it")
    win = _gen(cfg, sd, z[:, :, T - C - 5:], g)[:, C * hop:]
    assert float((win - w_full[:, (T - 5) * hop:]).abs().max()) < 1e-10
