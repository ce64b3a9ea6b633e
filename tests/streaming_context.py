"""Streaming windows of the flow and the decoder: the context each side that makes a window exact, restated in Python
from the module configurations (the library derives the same numbers from the pack's config: vsg_window_context)."""
from __future__ import annotations


def flow_context(cfg) -> int:
    """Frames each side that one output frame of ResidualCouplingBlock (either direction) depends on: every coupling layer's
    WaveNet (in_layers of kernel_size at dilation_rate**i, padding (k*d - d) / 2; pre / post are 1x1)."""
    r, dil = 0, 1
    for _ in range(cfg["n_layers"]):
        k = cfg["kernel_size"]
        pad = (k * dil - dil) // 2
        r += max(pad, (k - 1) * dil - pad)
        dil *= cfg["dilation_rate"]
    return r * cfg["n_flows"]


def dec_context(cfg) -> int:
    """Frames each side a window of the Generator needs: the receptive field of output frame 0 walked back through
    conv_post, each stage's resblocks (the widest of its parallel blocks) and upsampler, and conv_pre, noting at every
    rate the latent frames its samples lie in (a window's tensor at that rate covers whole frames)."""
    ur, uk = cfg["ur"], cfg["uk"]
    hop = 1
    for r in ur:
        hop *= r
    R, lo, hi = hop, 0, hop - 1
    left = right = 0

    def note():
        nonlocal left, right
        left = max(left, -(lo // R))
        right = max(right, hi // R)

    def conv(k, d):
        nonlocal lo, hi
        pad = (k * d - d) // 2
        lo -= pad
        hi += (k - 1) * d - pad

    conv(7, 1)                                     # conv_post
    note()
    for i in reversed(range(len(ur))):
        rlo = rhi = 0
        for k, ds in zip(cfg["rk"], cfg["rd"]):
            lo0, hi0 = lo, hi
            for d in reversed(ds):
                if str(cfg["resblock"]) == "1":
                    conv(k, 1)
                conv(k, d)
            rlo, rhi = min(rlo, lo - lo0), max(rhi, hi - hi0)
            lo, hi = lo0, hi0
        lo, hi = lo + rlo, hi + rhi
        note()
        r, k = ur[i], uk[i]
        pad = (k - r) // 2
        lo = -((-(lo + pad - k + 1)) // r)         # ceil
        hi = (hi + pad) // r
        R //= r
        note()
    conv(7, 1)                                     # conv_pre
    note()
    return max(left, right)
