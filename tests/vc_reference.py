"""Float64 references of voice conversion (VISinger.voice_conversion / vsg_model_convert) on the CPU.

`linear_spectrogram` states the posterior encoder's input: VITS's spectrogram_torch of each utterance on its own, on
torch.stft in float64.  `direct_spectrogram` is an independent statement of the same sum (an explicit DFT, optionally on
operands rounded as the bf16 kernel sees them), and `voice_conversion` composes the oracle's posterior encoder, flow (both
directions) and generator."""
import math
from typing import Optional

import numpy as np
import torch

from oracle import visinger_oracle as O


def reflect_index(idx: torch.Tensor, length: int) -> torch.Tensor:
    """torch's 'reflect' padding as an index map onto [0, length): no edge repeat, folded again while outside."""
    if length <= 1:
        return torch.zeros_like(idx)
    per = 2 * (length - 1)
    m = torch.remainder(idx, per)
    return torch.where(m < length, m, per - m)


def linear_spectrogram(wav, lengths, *, n_fft: int, hop: int, win_length: Optional[int] = None) -> torch.Tensor:
    """Reflect pad (n_fft - hop) // 2 about the utterance's own ends, periodic Hann window of win_length centred in n_fft,
    torch.stft(center=False), sqrt(|X|^2 + 1e-6), per utterance, in float64.  wav [B, T * hop]; utterance b is its first
    lengths[b] * hop samples (lengths clamped to [0, T]).  Returns [B, n_fft // 2 + 1, T], zero on frames t >= lengths[b]."""
    wav = torch.as_tensor(wav).to(torch.float64)
    B, L = wav.shape
    T = L // hop
    win = win_length or n_fft
    p = (n_fft - hop) // 2
    window = torch.hann_window(win, periodic=True, dtype=torch.float64)
    out = torch.zeros(B, n_fft // 2 + 1, T, dtype=torch.float64)
    for b in range(B):
        n = min(max(int(lengths[b]), 0), T)
        if n == 0:
            continue
        idx = reflect_index(torch.arange(-p, (n - 1) * hop - p + n_fft), n * hop)
        X = torch.stft(wav[b, idx], n_fft, hop_length=hop, win_length=win, window=window, center=False,
                       return_complex=True)
        out[b, :, :n] = torch.sqrt(X.real ** 2 + X.imag ** 2 + 1e-6)[:, :n]
    return out


def spectrogram_torch(y, *, n_fft: int, hop: int, win_length: int) -> torch.Tensor:
    """VITS mel_processing.spectrogram_torch (center=False), in float64: y [B, L] -> [B, n_fft // 2 + 1, frames]."""
    y = torch.as_tensor(y).to(torch.float64)
    pad = int((n_fft - hop) / 2)
    y = torch.nn.functional.pad(y.unsqueeze(1), (pad, pad), mode="reflect").squeeze(1)
    X = torch.stft(y, n_fft, hop_length=hop, win_length=win_length,
                   window=torch.hann_window(win_length, dtype=torch.float64), center=False, return_complex=True)
    return torch.sqrt(X.real ** 2 + X.imag ** 2 + 1e-6)


def _bf16(x: np.ndarray) -> np.ndarray:
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16).to(torch.float64).numpy()


def direct_spectrogram(wav, lengths, *, n_fft: int, hop: int, win_length: int, bf16: bool = False):
    """The same statement as an explicit DFT sum, frame by frame (no torch.stft).  bf16=True evaluates it on the operands
    the tcgen05 kernel multiplies: samples rounded to bf16, and the window-folded basis w[n] cos / -w[n] sin evaluated in
    double, rounded to fp32 and then to bf16.  Returns (spec [B, bins, T], S [B, T]) with S = sum_n |w[n] y[n]| of each
    frame (the scale of the rounding errors), both float64 and zero beyond lengths."""
    wav = np.asarray(torch.as_tensor(wav), dtype=np.float64)
    B, L = wav.shape
    T, bins, p, lead = L // hop, n_fft // 2 + 1, (n_fft - hop) // 2, (n_fft - win_length) // 2
    nr = np.arange(win_length)
    w = 0.5 - 0.5 * np.cos(2 * math.pi * nr / win_length)
    n = lead + nr
    phase = 2 * math.pi * ((np.arange(bins)[:, None] * n[None, :]) % n_fft) / n_fft
    re_b, im_b = w * np.cos(phase), -w * np.sin(phase)                                   # [bins, win]
    if bf16:
        re_b, im_b = _bf16(re_b.astype(np.float32)), _bf16(im_b.astype(np.float32))
    spec, S = np.zeros((B, bins, T)), np.zeros((B, T))
    for b in range(B):
        m = min(max(int(lengths[b]), 0), T)
        if m == 0:
            continue
        y = wav[b].astype(np.float32).astype(np.float64)
        if bf16:
            y = _bf16(y)
        idx = reflect_index(torch.arange(m)[:, None] * hop - p + torch.from_numpy(n)[None, :], m * hop).numpy()
        fr = y[idx]                                                                        # [m, win]
        re, im = fr @ re_b.T, fr @ im_b.T
        spec[b, :, :m] = np.sqrt(re ** 2 + im ** 2 + 1e-6).T
        S[b, :m] = np.abs(fr * w[None, :]).sum(1)
    return spec, S


def voice_conversion(sd, spec, mask, g_src, g_tgt, noise, *, post_kw=None, flow_kw=None, dec_kw=None):
    """VITS SynthesizerTrn.voice_conversion on VISinger's modules, from the oracle's pieces:
    z = posterior(spec, g_src); z_p = flow(z, g_src); z_hat = flow(z_p, g_tgt, reverse) * mask;
    wav = decoder(z_hat * mask, g_tgt).  Returns (wav [B, L], z_hat)."""
    z, _, _ = O.posterior_encoder(sd, spec, mask, g_src, noise, prefix="posterior_encoder.", **(post_kw or {}))
    z_p = O.flow(sd, z, mask, g=g_src, reverse=False, prefix="flow.", **(flow_kw or {}))
    z_hat = O.flow(sd, z_p, mask, g=g_tgt, reverse=True, prefix="flow.", **(flow_kw or {})) * mask
    wav = O.generator(sd, z_hat * mask, g=g_tgt, prefix="decoder.", **(dec_kw or {})).squeeze(1)
    return wav, z_hat
