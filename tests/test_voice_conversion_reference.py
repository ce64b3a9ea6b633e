"""The float64 statement of the linear spectrogram (tests/vc_reference.py) and the convert calls' argument checks, on the
CPU.  linear_spectrogram (torch.stft, reflect index map) equals an explicit DFT sum, including utterances so short that the
padding folds more than once; with full lengths and even n_fft - hop it equals VITS's spectrogram_torch of the utterance."""
import ctypes

import numpy as np
import pytest
import torch

from model_inputs import SMALL_HPARAMS
from vc_reference import direct_spectrogram, linear_spectrogram, reflect_index, spectrogram_torch

VSG_EINVAL = -1


def _wav(seed, B, L):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(L, dtype=torch.float64)
    f = 0.01 + 0.2 * torch.rand(B, 1, generator=g, dtype=torch.float64)
    return (0.5 * torch.sin(f * t) + 0.1 * torch.randn(B, L, generator=g, dtype=torch.float64)).float()


def test_reflect_index_matches_torch_reflect_pad():
    x = torch.arange(7, dtype=torch.float64)[None, None]
    ref = torch.nn.functional.pad(x, (6, 6), mode="reflect")[0, 0]
    assert torch.equal(x[0, 0, reflect_index(torch.arange(-6, 13), 7)], ref)
    # folded again beyond one length: a period of 2 (L - 1)
    assert reflect_index(torch.tensor([-13, 13, 20]), 7).tolist() == [1, 1, 4]
    assert reflect_index(torch.tensor([-3, 0, 5]), 1).tolist() == [0, 0, 0]


@pytest.mark.parametrize("n_fft,hop,win", [(64, 15, 60), (64, 15, 64), (64, 16, 60), (2048, 300, 1200)])
def test_linear_spectrogram_equals_direct_dft(n_fft, hop, win):
    T = 9 if n_fft > 64 else 40
    lengths = [T, 1, 2, 5] if n_fft > 64 else [T, 1, 2, 3, 17]
    wav = _wav(1, len(lengths), T * hop)
    a = linear_spectrogram(wav, lengths, n_fft=n_fft, hop=hop, win_length=win)
    b, S = direct_spectrogram(wav, lengths, n_fft=n_fft, hop=hop, win_length=win)
    err = (a.numpy() - b).max(axis=1)
    assert np.all(np.abs(err) <= 1e-12 * np.maximum(S, 1.0))
    for i, n in enumerate(lengths):
        assert torch.all(a[i, :, n:] == 0)


@pytest.mark.parametrize("n_fft,hop,win", [(64, 16, 60), (64, 16, 64), (2048, 300, 1200)])
def test_linear_spectrogram_equals_spectrogram_torch_on_full_lengths(n_fft, hop, win):
    T = 7 if n_fft > 64 else 30
    wav = _wav(2, 3, T * hop)
    a = linear_spectrogram(wav, [T] * 3, n_fft=n_fft, hop=hop, win_length=win)
    b = spectrogram_torch(wav, n_fft=n_fft, hop=hop, win_length=win)
    assert b.shape == a.shape
    torch.testing.assert_close(a, b, rtol=0, atol=1e-12)
    # and on the utterance alone: a shorter utterance of the batch is spectrogram_torch of its own samples
    n = 4 if n_fft > 64 else 11
    c = linear_spectrogram(wav, [n, T, T], n_fft=n_fft, hop=hop, win_length=win)
    torch.testing.assert_close(c[0, :, :n], spectrogram_torch(wav[:1, :n * hop], n_fft=n_fft, hop=hop, win_length=win)[0],
                               rtol=0, atol=1e-12)


def _small_cfg_and_weights(drop=None, bins=33):
    from visinger_b200.models.visinger import VISinger
    from visinger_b200 import _lib
    torch.manual_seed(0)
    m = VISinger(73, 117, 132, dict(SMALL_HPARAMS))
    sd = {k: v for k, v in m.state_dict().items() if k != drop}
    if bins != 33:
        sd["posterior_encoder.pre.weight"] = torch.zeros(32, bins, 1)
    arr, keep = _lib._weight_table({k: v.float().contiguous() for k, v in sd.items()})
    return m._model_config(), arr, len(keep), (sd, keep)


def test_convert_calls_reject_bad_arguments_without_gpu():
    from visinger_b200 import _lib
    L = _lib.lib()
    out = ctypes.c_void_p()
    assert L.vsg_convert_pack_create(None, None, 0, b"", 64, 0, ctypes.byref(out)) == VSG_EINVAL and not out.value
    cfg, arr, n, keep = _small_cfg_and_weights(drop="posterior_encoder.pre.weight")
    rc = L.vsg_convert_pack_create(ctypes.byref(cfg), arr, n, b"", 64, 0, ctypes.byref(out))
    assert rc == VSG_EINVAL and b"posterior_encoder.pre.weight" in L.vsg_last_error()
    cfg, arr, n, keep = _small_cfg_and_weights()
    for win in (0, 65, -3):          # n_fft = 2 * (33 - 1) = 64
        rc = L.vsg_convert_pack_create(ctypes.byref(cfg), arr, n, b"", win, 0, ctypes.byref(out))
        assert rc == VSG_EINVAL and b"win_length" in L.vsg_last_error() and not out.value
    cfg, arr, n, keep = _small_cfg_and_weights(bins=8)   # n_fft 14 < hop 15
    rc = L.vsg_convert_pack_create(ctypes.byref(cfg), arr, n, b"", 14, 0, ctypes.byref(out))
    assert rc == VSG_EINVAL and b"hop" in L.vsg_last_error()
    assert L.vsg_convert_workspace_bytes(None, 1, 8, 0) == 0
    args = [None] * 13 + [1, 8, 0, None, 0, None]
    assert L.vsg_model_convert(*args) == VSG_EINVAL and L.vsg_last_launch_count() == 0
    assert L.vsg_spectrogram(None, None, None, None, 1, 8, 0, None, 0, None) == VSG_EINVAL
    assert L.vsg_last_launch_count() == 0


def test_voice_conversion_refuses_cpu_tensors():
    from visinger_b200.models.visinger import VISinger
    m = VISinger(73, 117, 132, dict(SMALL_HPARAMS))
    with pytest.raises(RuntimeError, match="CPU fallback|CUDA"):
        m.voice_conversion(wav=torch.zeros(1, 150), lengths=torch.tensor([10]), spk_id=[0], tgt_spk_id=[1])
