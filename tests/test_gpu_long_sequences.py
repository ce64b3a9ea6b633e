"""Utterances longer than 2048 latent frames through the prior network.

The bf16 encoder's attention splits the keys into chunks of at most 2048 beyond T = 2048 (csrc/attn_tc.cuh, split-key
mode): each CTA runs the two-pass softmax over one key chunk and writes unnormalised partials, and a combine kernel merges
the chunks.  `debug_attention_split_bf16` runs that path at any T and any key chunk that is a multiple of 128, so small T
can cover many chunks.  It is held to the float64 statement and gates of test_gpu_attention.py: (a) against the exact
operation; (b) against the same with P rounded to bf16 relative to each chunk's own maximum, as the kernel rounds it.
Beside the tolerances: one chunk equals the single launch bit for bit, masked padding and batching leave the bits
unchanged, and repeated runs give the same bits.  Then the whole RelativeEncoder, the length regulator past its old
12 288-frame limit, and a whole VISinger.forward on a 4600-frame utterance in all three modes."""
import math

import pytest
import torch

from oracle import visinger_oracle as O
from helpers import maxabs
from test_gpu_attention import (BF, HEADS, WINDOWS, TOL_A_MAX, TOL_A_MEAN, TOL_B_MAX, TOL_B_MEAN, TOL_BORDER_RATIO,
                                attention_fp64, _inputs, _masks, _split, _heads, _rel, _run_bf16, _border_ratio)

pytestmark = pytest.mark.gpu

# Measured on a B200 (1000 W) over the split-attention cases below: (a) max 8.6e-3, mean 7.9e-4; (b) max 4.3e-3, mean
# 6.4e-4; chunk-border rows over the others 0.84 .. 1.10 -- inside the gates of test_gpu_attention.py, which apply as they are.


def _run_split(qkv, mask, ek, ev, heads, d, key_chunk=0):
    from visinger_b200 import _lib
    return _lib.debug_attention_split_bf16(qkv.to(d), mask.to(d), ek.to(d), ev.to(d), heads, key_chunk)


def attention_fp64_chunked_p(q, k, v, mask, ek, ev, w, chunk):
    """attention_fp64 with P rounded to bf16 relative to the maximum of its own key chunk (chunks of `chunk` keys from
    key 0), the chunks then weighted by exp(m_c - M) as the combine does.  Row sums and relative-value weights unrounded."""
    T, dk = q.shape[2], q.shape[3]
    i = torch.arange(T, device=q.device)
    offset = i[None, :] - i[:, None]
    bands = [(offset == r - w).to(q.dtype) for r in range(2 * w + 1)]
    s = q @ k.transpose(-1, -2)
    qe = q @ ek.t()
    for r, band in enumerate(bands):
        s = s + qe[..., r:r + 1] * band
    s = s / math.sqrt(dk)
    pair = mask[:, None, :, None] * mask[:, None, None, :]
    s = s.masked_fill(pair == 0, -1e4)
    n_chunks = (T + chunk - 1) // chunk
    m_c = torch.stack([s[..., c * chunk:(c + 1) * chunk].amax(-1) for c in range(n_chunks)], -1)   # [B, h, T, chunks]
    mcol = m_c[..., i // chunk]                                                                    # [B, h, T, T]
    e = torch.exp(s - mcol)
    del s
    wcol = torch.exp(mcol - m_c.amax(-1, keepdim=True))
    del mcol
    o = (e.to(BF).to(q.dtype) * wcol) @ v
    e = e * wcol
    for r, band in enumerate(bands):
        o = o + (e * band).sum(-1, keepdim=True) * ev[r]
    return o / e.sum(-1, keepdim=True)


def _check_split_case(d, dk, heads, w, T, key_chunk, seed):
    mask = _masks(T, seed)
    chunk = key_chunk or 2048
    for peaky in (True, False):
        qkv, ek, ev = _inputs(mask.shape[0], T, heads, dk, w, peaky, seed + peaky)
        o = _heads(_run_split(qkv, mask, ek, ev, heads, d, key_chunk), heads, dk)
        q, k, v = (t.to(d) for t in _split(qkv, heads, dk))
        args = (q, k, v, mask.double().to(d), ek.to(BF).double().to(d), ev.double().to(d), w)
        rel_a = _rel(o, attention_fp64(*args))
        rel_b = _rel(o, attention_fp64_chunked_p(*args, chunk))
        ratio = _border_ratio(rel_b, mask, T, w, chunk) if w > 0 else None
        print(f"split attention dk={dk} h={heads} w={w} T={T} chunk={chunk} {'peaky' if peaky else 'flat'}: "
              f"(a) max {float(rel_a.max()):.2e} mean {float(rel_a.mean()):.2e}  (b) max {float(rel_b.max()):.2e} "
              f"mean {float(rel_b.mean()):.2e}  chunk-border rms ratio {'-' if ratio is None else f'{ratio:.2f}'}")
        assert torch.isfinite(o).all()
        assert float(rel_a.max()) <= TOL_A_MAX and float(rel_a.mean()) <= TOL_A_MEAN
        assert float(rel_b.max()) <= TOL_B_MAX and float(rel_b.mean()) <= TOL_B_MEAN
        assert ratio is None or ratio <= TOL_BORDER_RATIO
        del rel_a, rel_b, o
        torch.cuda.empty_cache()


@pytest.mark.parametrize("dk,heads", HEADS)
@pytest.mark.parametrize("w", WINDOWS)
@pytest.mark.parametrize("T", [257, 300])
def test_split_attention_small_chunks_every_width_and_window(cuda_device, dk, heads, w, T):
    """Chunks of 128 keys: three chunks, the last ragged (T = 257: one key), and windows across two chunk borders."""
    _check_split_case(cuda_device, dk, heads, w, T, 128, dk * 31 + heads * 7 + w + T)


LONG = [2049, 2050, 4095, 4096, 4097, 6000]


@pytest.mark.parametrize("T", LONG)
def test_split_attention_default_chunks(cuda_device, T):
    """The encoder's chunks of 2048 keys just past each chunk-count edge; head configuration and window rotate."""
    i = LONG.index(T)
    dk, heads = HEADS[(3 * i + 1) % len(HEADS)]
    _check_split_case(cuda_device, dk, heads, WINDOWS[(i + 1) % len(WINDOWS)], T, 0, 2000 + T)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,dk,heads,w", [(1, 16, 4, 0), (129, 32, 2, 1), (1000, 48, 4, 7), (2048, 64, 2, 4),
                                          (2047, 96, 2, 4)])
def test_split_attention_one_chunk_equals_single_launch(cuda_device, T, dk, heads, w):
    """At T <= 2048 the split path with one chunk gives the single launch's bits: the chunk's weight is exactly 1."""
    mask = _masks(T, T)
    qkv, ek, ev = _inputs(mask.shape[0], T, heads, dk, w, True, T + 5)
    assert torch.equal(_run_split(qkv, mask, ek, ev, heads, cuda_device), _run_bf16(qkv, mask, ek, ev, heads, cuda_device))


@pytest.mark.parametrize("n,T,key_chunk", [(1000, 2100, 0), (2048, 4097, 0), (1500, 6000, 0), (2500, 4500, 0),
                                           (4096, 6200, 0), (200, 300, 128), (129, 640, 128), (300, 1000, 256)])
def test_split_attention_padding_is_exact(cuda_device, n, T, key_chunk):
    """One utterance of n frames alone (T = n) and padded into T frames with large masked garbage beyond n: the n valid
    rows are identical bit for bit.  Chunks past n hold only masked keys: their weight in the combine is exactly 0 and
    their partial output finite.  Where the alone run is one chunk of the default size, it equals the single launch."""
    dk, heads, w = 64, 2, 4
    qkv, ek, ev = _inputs(1, T, heads, dk, w, n % 2 == 0, 7 * n + T)
    gen = torch.Generator().manual_seed(n)
    qkv[:, n:] = ((torch.rand(1, T - n, qkv.shape[2], generator=gen) * 2 - 1) * 3e4).to(BF)
    mask = torch.ones(1, T)
    mask[:, n:] = 0
    alone_qkv = qkv[:, :n].contiguous()
    alone = _run_split(alone_qkv, torch.ones(1, n), ek, ev, heads, cuda_device, key_chunk)
    padded = _run_split(qkv, mask, ek, ev, heads, cuda_device, key_chunk)
    assert torch.isfinite(padded.float()).all()
    assert torch.equal(alone, padded[:, :n])
    if key_chunk == 0 and n <= 2048:
        assert torch.equal(alone, _run_bf16(alone_qkv, torch.ones(1, n), ek, ev, heads, cuda_device))


@pytest.mark.parametrize("T,key_chunk", [(385, 128), (2500, 0)])
def test_split_attention_batch_invariant_and_deterministic(cuda_device, T, key_chunk):
    """Each utterance of a six-utterance batch gives the bits it gives alone; a second run gives the same bits."""
    dk, heads, w = 16, 4, 4
    mask = _masks(T, T)
    qkv, ek, ev = _inputs(mask.shape[0], T, heads, dk, w, True, T)
    o = _run_split(qkv, mask, ek, ev, heads, cuda_device, key_chunk)
    assert torch.equal(o, _run_split(qkv, mask, ek, ev, heads, cuda_device, key_chunk))
    for b in range(mask.shape[0]):
        alone = _run_split(qkv[b:b + 1].contiguous(), mask[b:b + 1], ek, ev, heads, cuda_device, key_chunk)
        assert torch.equal(alone, o[b:b + 1])


def test_split_attention_rejects_bad_key_chunks(cuda_device):
    """A key chunk that is not a multiple of 128 between 128 and 2048 (or 0) is refused with VSG_EINVAL."""
    qkv, ek, ev = _inputs(1, 300, 2, 32, 4, False, 9)
    for kc in (64, 200, 2176, -128):
        with pytest.raises(RuntimeError) as e:
            _run_split(qkv, torch.ones(1, 300), ek, ev, 2, cuda_device, kc)
        assert "failed (-1)" in str(e.value), str(e.value)                 # VSG_EINVAL


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [2049, 4500])
def test_relenc_bf16_long_vs_oracle(cuda_device, T):
    """The bf16 RelativeEncoder (hidden 192, 2 heads, window 4) beyond 2048 frames, one ragged utterance, at the gates of
    the full-config bf16 test in test_relenc.py; masked frames exactly 0."""
    from visinger_b200.modules.rel_transformer import RelativeEncoder
    cfg = dict(hidden=192, filter=768, n_heads=2, n_layers=2, kernel_size=9, window=4, gin=16)
    sd = O.synth_rel_encoder_state_dict(O.rel_encoder_param_shapes(192, 768, 2, 2, 9, 4, 16), T)
    gen = torch.Generator().manual_seed(T + 1)
    x, g = torch.randn(2, 192, T, generator=gen), torch.randn(2, 16, 1, generator=gen)
    mask = torch.ones(2, 1, T)
    mask[1, :, T * 3 // 5:] = 0
    with torch.no_grad():
        yo = O.rel_encoder(sd, x, mask, g, n_heads=2, n_layers=2, kernel_size=9, window=4)
    m = RelativeEncoder(192, 768, 2, 2, kernel_size=9, window_size=4, gin_channels=16)
    m.load_state_dict(sd, strict=True)
    m = m.to(cuda_device).eval()
    m.precision = "bf16"
    y = m(x.to(cuda_device), mask.to(cuda_device), g.to(cuda_device)).cpu()
    rel = float((y - yo).norm() / yo.norm())
    print(f"relenc bf16 T={T} ({cfg}): rel-L2 {rel:.3e} max-abs {maxabs(y, yo):.3e}")
    assert rel <= 8.5e-3 and maxabs(y, yo) <= 0.09
    assert float((y * (1 - mask)).abs().max()) == 0.0


@pytest.mark.parametrize("T", [12289, 30000])
@pytest.mark.parametrize("use_pos", [True, False])
def test_length_regulate_long(cuda_device, T, use_pos):
    """Beyond the 12 288 frames the one-pass kernel held in shared memory: bit-exact against the reference formula."""
    from visinger_b200 import _lib
    from test_prior_head import _regulate_ref, _sin_table, _mel2ph
    B, H, T_ph = 2, 192, 400
    gen = torch.Generator().manual_seed(T + use_pos)
    enc = torch.randn(B, H, T_ph, generator=gen)
    enc[0, 0, 5] = 0.0                                  # frames of a token whose channel 0 is zero get no position
    lengths = [T, T - 4321]
    mel2ph = _mel2ph(B, T_ph, T, gen, lengths)
    table = _sin_table(T + 1, H) if use_pos else None
    want = _regulate_ref(enc, mel2ph, table)
    got = _lib.length_regulate(enc.to(cuda_device), mel2ph.to(cuda_device), table.to(cuda_device) if use_pos else None)
    assert torch.equal(got.cpu(), want)


# ---------------------------------------------------------------------------------------------------------------------
LENGTHS = [4600, 900]


@pytest.fixture(scope="module")
def long_song():
    """A batch of two utterances (4600 and 900 frames, right-padded), injected noise, and the CPU reference: the seeded
    full-hparams mirror's PyTorch prior() on the CPU, then the oracle's flow reverse and decoder."""
    from model_inputs import full_model_mirror, synth_utterances
    m = full_model_mirror()
    batch = synth_utterances(seed=4600, n=2, lengths=LENGTHS)
    T = batch["mel2ph"].shape[1]
    noise = torch.randn(2, 192, T, generator=torch.Generator().manual_seed(46))
    ret = {}
    with torch.no_grad():
        mu, logs, mask, spk = m.prior(batch["text_tokens"], batch["note_pitch"], batch["note_dur"], batch["mel2ph"],
                                      spk_id=batch["spk_ids"], ret=ret)
        sd = {k: v for k, v in m.state_dict().items() if k.startswith(("flow.", "decoder."))}
        wav_ref, _ = O.infer_hot_path(sd, mu, logs, noise, mask, spk)
    return batch, noise, wav_ref, ret["f0_pred"]


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_visinger_forward_long_utterance(cuda_device, long_song, precision):
    """Whole forward(infer=True) on a 4600-frame utterance (1.38 M samples at hop 300) and a 900-frame one, against the
    CPU reference over the whole waveform, padded region included, at the gates of the config-4 test.  bf16:
    forward_graphed at this shape equals the eager forward bit for bit."""
    from model_inputs import full_model_mirror
    batch, noise, wav_ref, f0_ref = long_song
    m = full_model_mirror(precision=precision).to(cuda_device)            # the reference's weights (same seed)
    d = {k: v.to(cuda_device) for k, v in batch.items()}
    args = (d["text_tokens"], d["note_pitch"], d["note_dur"], d["mel2ph"])
    out = m(*args, spk_id=d["spk_ids"], infer=True, noise=noise.to(cuda_device))
    wav = out["wav_out"].cpu()
    assert wav.shape == wav_ref.shape
    err = maxabs(wav, wav_ref)
    rel = float((wav - wav_ref).norm() / wav_ref.norm())
    e_f0 = maxabs(out["f0_pred"].cpu(), f0_ref)
    print(f"VISinger forward T={LENGTHS} {precision}: waveform max-abs {err:.3e} (|ref|max {float(wav_ref.abs().max()):.3e}), "
          f"rel-L2 {rel:.3e}, f0 {e_f0:.3e}")
    if precision == "bf16":
        assert rel <= 3e-2 and err <= 5e-3
        got = m.forward_graphed(*args, spk_id=d["spk_ids"], noise=noise.to(cuda_device))
        assert torch.equal(got["wav_out"], out["wav_out"]) and torch.equal(got["f0_pred"], out["f0_pred"])
    else:
        assert err <= 1e-4 and e_f0 <= 5e-5
