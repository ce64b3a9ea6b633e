"""The relative-position encoder's attention kernels one at a time, against a float64 statement of
MultiHeadAttention.attention (modules/rel_transformer.py:137-177: windowed, heads_share=True):

    s_ij = (q_i . k_j + [|j-i| <= w] q_i . Ek[j-i+w]) / sqrt(dk);  s_ij = -1e4 where mask_i * mask_j == 0
    o_i  = sum_j softmax_j(s)_ij (v_j + [|j-i| <= w] Ev[j-i+w])

The bf16 tcgen05 kernel (csrc/attn_tc.cuh) is compared with two references: (a) the same operation in float64 from the
operands the kernel sees (q, k, v and Ek rounded to bf16, Ev fp32), a loose bound on its total error; (b) the same with P
rounded to bf16 before P V, as the kernel does (row sums and relative-value weights unrounded), which leaves fp32
accumulation order, exp2f and the final bf16 rounding of o.  Errors are measured relative to the largest |o| of each output
row, so rows of small magnitude (masked query rows, flat softmax over long sequences) are held to the same standard.
Beside the tolerances: padding invariance and batch invariance bit for bit, determinism, and the error of query rows whose
window crosses a 32-column chunk or a 128-row tile border against the other rows.  The fp32 kernel (csrc/relenc_f32.cuh)
is compared with (a) unrounded."""
import math

import pytest
import torch

BF = torch.bfloat16
gpu = pytest.mark.gpu

# (head width, heads): every instantiated width with H = heads * dk <= 256 (dk = 128 is rejected: test below)
HEADS = [(16, 1), (16, 4), (32, 2), (32, 4), (48, 1), (48, 4), (64, 2), (64, 4), (96, 1), (96, 2)]
WINDOWS = [0, 1, 4, 7]
# 1 .. 16 key tiles: odd and even counts, nt = 1 (softmax set 0 has no pass-2 visit), ragged and full last tiles
LENGTHS = [1, 2, 31, 33, 127, 128, 129, 255, 256, 257, 1000, 2047, 2048]

# Gates, relative to the row's largest |o|, at 1.5-2x the largest value measured over all cases of this file on a B200
# (1000 W): (a) max 7.4e-3, mean 8.3e-4; (b) max 4.1e-3 (the final bf16 rounding of o alone reaches 2^-8 = 3.9e-3), mean
# 6.2e-4; window-crossing rows over the others 0.89 .. 1.13; fp32 kernel max 4.5e-6.  TOL_B_MAX is one bf16 ulp of |o|.
TOL_A_MAX, TOL_A_MEAN = 1.5e-2, 1.5e-3
TOL_B_MAX, TOL_B_MEAN = 2 ** -7, 1.0e-3
TOL_F32_MAX = 1e-5
TOL_BORDER_RATIO = 1.7


# ---------------------------------------------------------------------------------------------------------------------
# float64 statement of the operation: dense band matrices, one per relative offset (the oracle gathers / scatters, the
# module uses diagonal views)
def attention_fp64(q, k, v, mask, ek, ev, w, p_bf16=False):
    """q, k, v: [B, h, T, dk]; mask: [B, T]; ek, ev: [2w+1, dk]; float64 on any device.  p_bf16: round the unnormalised
    probabilities to bf16 for P V only, as the tensor-core kernel does.  Returns o [B, h, T, dk]."""
    T, dk = q.shape[2], q.shape[3]
    i = torch.arange(T, device=q.device)
    offset = i[None, :] - i[:, None]                                   # j - i
    bands = [(offset == r - w).to(q.dtype) for r in range(2 * w + 1)]
    s = q @ k.transpose(-1, -2)
    qe = q @ ek.t()                                                    # [B, h, T, 2w+1]
    for r, band in enumerate(bands):
        s = s + qe[..., r:r + 1] * band
    s = s / math.sqrt(dk)
    pair = mask[:, None, :, None] * mask[:, None, None, :]
    s = s.masked_fill(pair == 0, -1e4)
    e = torch.exp(s - s.amax(-1, keepdim=True))
    pv = e.to(BF).to(q.dtype) if p_bf16 else e
    o = pv @ v
    for r, band in enumerate(bands):
        o = o + (e * band).sum(-1, keepdim=True) * ev[r]
    return o / e.sum(-1, keepdim=True)


def _conv(x, m, name):
    conv = getattr(m, name)
    return torch.nn.functional.conv1d(x, conv.weight, conv.bias)


def test_fp64_statement_matches_the_module_and_the_oracle():
    """CPU: the statement above inside MultiHeadAttention.forward (projections and conv_o around it) equals the module's
    diagonal-view formulation and the oracle's gather / scatter one, with a ragged mask, at T below and above 2w+1."""
    from oracle import visinger_oracle as O
    from visinger_b200.modules.rel_transformer import MultiHeadAttention
    torch.manual_seed(0)
    for T, w, heads, C in ((13, 4, 2, 16), (5, 4, 1, 8), (40, 1, 4, 32)):
        m = MultiHeadAttention(C, C, heads, window_size=w).double().eval()
        with torch.no_grad():
            for prm in m.parameters():
                prm.copy_(torch.randn_like(prm))
        x = torch.randn(2, C, T, dtype=torch.float64)
        mask = torch.ones(2, T, dtype=torch.float64)
        mask[1, T - 3:] = 0
        mask[1, 1] = 0
        attn_mask = mask[:, None, :, None] * mask[:, None, None, :]
        with torch.no_grad():
            want = m(x, x, attn_mask)
            sd = {k: v for k, v in m.state_dict().items()}
            oracle = O.rel_attention(sd, "", x, attn_mask, n_heads=heads, window=w)
            dk = C // heads
            q, k, v = (_conv(x, m, n).view(2, heads, dk, T).transpose(2, 3) for n in ("conv_q", "conv_k", "conv_v"))
            o = attention_fp64(q, k, v, mask, m.emb_rel_k[0], m.emb_rel_v[0], w)
            got = torch.nn.functional.conv1d(o.transpose(2, 3).reshape(2, C, T), m.conv_o.weight, m.conv_o.bias)
        assert float((got - want).abs().max()) <= 1e-12 * float(want.abs().max())
        assert float((got - oracle).abs().max()) <= 1e-12 * float(want.abs().max())


# ---------------------------------------------------------------------------------------------------------------------
def _inputs(B, T, heads, dk, w, peaky, seed):
    """Channels-last bf16 qkv [B, T, 3H] as the fused projection writes it, and O(1) Ek / Ev.  Peaky: logits q.k / sqrt(dk)
    of standard deviation 8 (row maxima about 25-30); flat: 0.09, where the relative-position logits (std 0.3) dominate."""
    gen = torch.Generator().manual_seed(seed)
    H = heads * dk
    sig = 8 ** 0.5 if peaky else 0.3
    q = torch.randn(B, T, H, generator=gen) * sig
    k = torch.randn(B, T, H, generator=gen) * sig
    v = torch.randn(B, T, H, generator=gen)
    ek = torch.randn(2 * w + 1, dk, generator=gen)
    ev = torch.randn(2 * w + 1, dk, generator=gen)
    return torch.cat([q, k, v], -1).to(BF), ek, ev


def _masks(T, seed):
    """Six utterances: full, lengths 0, 1, 128 and 256 (clipped to T), and a non-prefix mask with holes."""
    gen = torch.Generator().manual_seed(seed)
    mask = torch.ones(6, T)
    for b, n in enumerate((0, 1, 128, 256)):
        mask[b + 1, min(n, T):] = 0
    mask[5] = (torch.rand(T, generator=gen) < 0.75).float()
    return mask


def _split(qkv, heads, dk):
    """[B, T, 3H] -> q, k, v float64 [B, h, T, dk]."""
    B, T, _ = qkv.shape
    x = qkv.double().view(B, T, 3, heads, dk).permute(2, 0, 3, 1, 4)
    return x[0], x[1], x[2]


def _heads(o, heads, dk):
    B, T, _ = o.shape
    return o.double().view(B, T, heads, dk).transpose(1, 2)


def _rel(o, ref):
    """|o - ref| over the largest |ref| of each output row."""
    return (o - ref).abs() / ref.abs().amax(-1, keepdim=True).clamp_min(1e-6)


def _run_bf16(qkv, mask, ek, ev, heads, d):
    from visinger_b200 import _lib
    return _lib.debug_attention_bf16(qkv.to(d), mask.to(d), ek.to(d), ev.to(d), heads)


def _references(qkv, mask, ek, ev, heads, dk, w, d):
    q, k, v = (t.to(d) for t in _split(qkv, heads, dk))
    ek_b = ek.to(BF).double().to(d)                         # the kernel keeps Ek in shared memory as bf16
    args = (q, k, v, mask.double().to(d), ek_b, ev.double().to(d), w)
    return attention_fp64(*args), attention_fp64(*args, p_bf16=True)


def _border_ratio(rel_b, mask, T, w, period):
    """rms error of the valid query rows whose window [i-w, i+w] crosses a multiple of `period`, over the rms of the
    other valid rows (None when either set is empty)."""
    i = torch.arange(T, device=rel_b.device)
    border = (torch.div(i - w, period, rounding_mode="floor") != torch.div(i + w, period, rounding_mode="floor"))
    valid = mask.to(rel_b.device).bool()[:, None, :].expand(rel_b.shape[:3])
    row_ms = rel_b.pow(2).mean(-1)
    a, b = row_ms[valid & border], row_ms[valid & ~border]
    if a.numel() == 0 or b.numel() == 0:
        return None
    return float(a.mean().sqrt() / b.mean().sqrt().clamp_min(1e-30))


def _check_bf16_case(cuda_device, dk, heads, w, T, seed):
    mask = _masks(T, seed)
    for peaky in (True, False):
        qkv, ek, ev = _inputs(mask.shape[0], T, heads, dk, w, peaky, seed + peaky)
        o = _heads(_run_bf16(qkv, mask, ek, ev, heads, cuda_device), heads, dk)
        ref_a, ref_b = _references(qkv, mask, ek, ev, heads, dk, w, cuda_device)
        rel_a, rel_b = _rel(o, ref_a), _rel(o, ref_b)
        ratios = [_border_ratio(rel_b, mask, T, w, p) for p in (32, 128)] if w > 0 else [None, None]
        print(f"attention bf16 dk={dk} h={heads} w={w} T={T} {'peaky' if peaky else 'flat'}: "
              f"(a) max {float(rel_a.max()):.2e} mean {float(rel_a.mean()):.2e}  "
              f"(b) max {float(rel_b.max()):.2e} mean {float(rel_b.mean()):.2e}  border rms ratio "
              + " / ".join("-" if r is None else f"{r:.2f}" for r in ratios))
        assert torch.isfinite(o).all()
        assert float(rel_a.max()) <= TOL_A_MAX and float(rel_a.mean()) <= TOL_A_MEAN
        assert float(rel_b.max()) <= TOL_B_MAX and float(rel_b.mean()) <= TOL_B_MEAN
        for r in ratios:
            assert r is None or r <= TOL_BORDER_RATIO


@gpu
@pytest.mark.parametrize("dk,heads", HEADS)
@pytest.mark.parametrize("w", WINDOWS)
def test_attention_bf16_every_width_and_window(cuda_device, dk, heads, w):
    """Every head width and window at T = 257 (three key tiles, ragged last tile), ragged and holed masks."""
    _check_bf16_case(cuda_device, dk, heads, w, 257, dk * 31 + heads * 7 + w)


@gpu
@pytest.mark.parametrize("T", LENGTHS)
def test_attention_bf16_every_length(cuda_device, T):
    """Every tile-count edge, the head configuration and window rotating with the length."""
    i = LENGTHS.index(T)
    dk, heads = HEADS[(3 * i) % len(HEADS)]
    _check_bf16_case(cuda_device, dk, heads, WINDOWS[i % len(WINDOWS)], T, 1000 + T)


@gpu
@pytest.mark.parametrize("T", [1, 2, 31, 33, 127, 129, 200])
def test_attention_bf16_fully_masked_rows(cuda_device, T):
    """Masked query rows (a whole utterance of length 0, and the tail of a ragged one) are a uniform softmax over the T
    keys in the reference; the encoder carries them forward, so they are compared too, at the emulated-rounding gate.
    Their probabilities are all exactly 1, so the only error left is the sum order and the final rounding."""
    dk, heads, w = 32, 2, 4
    mask = torch.ones(2, T)
    mask[0] = 0
    mask[1, T // 2:] = 0
    qkv, ek, ev = _inputs(2, T, heads, dk, w, False, 77 + T)
    o = _heads(_run_bf16(qkv, mask, ek, ev, heads, cuda_device), heads, dk)
    _, ref_b = _references(qkv, mask, ek, ev, heads, dk, w, cuda_device)
    rel = _rel(o, ref_b)
    masked = (mask == 0).to(cuda_device)[:, None, :].expand(rel.shape[:3])
    print(f"attention bf16 masked rows T={T}: max {float(rel[masked].max()):.2e} (all rows {float(rel.max()):.2e})")
    assert float(rel.max()) <= TOL_B_MAX


@gpu
@pytest.mark.parametrize("n,T,dk,heads,w", [
    (1, 100, 64, 2, 4), (33, 127, 64, 2, 4), (100, 128, 64, 2, 4), (129, 250, 64, 2, 4), (700, 768, 64, 2, 4),
    (1000, 1024, 64, 2, 4), (2000, 2048, 64, 2, 4),                                    # same key-tile count
    (100, 300, 48, 4, 7), (128, 129, 48, 4, 7), (200, 300, 48, 4, 7), (129, 1000, 48, 4, 7), (1000, 2048, 48, 4, 7)])
def test_attention_bf16_padding_is_exact(cuda_device, n, T, dk, heads, w):
    """One utterance of n frames run alone (T = n) and inside a buffer of T frames, the frames past n holding large finite
    garbage and masked off: the n valid rows must be identical bit for bit.  Masked keys score -1e4 * log2(e), for which
    exp2f gives exactly 0, and 0 times a finite value adds nothing in the MMA.  This holds when T adds key tiles too: those
    tiles add exact zeros, P V accumulates in tile order whichever softmax set wrote P, and the two sets' row sums and
    relative-value weights are combined with one (commutative) add -- even where the extra tiles swap which set takes
    which valid tile (n = 200 in T = 300)."""
    qkv, ek, ev = _inputs(1, T, heads, dk, w, n % 2 == 0, 5 * n + T)
    gen = torch.Generator().manual_seed(n)
    qkv[:, n:] = ((torch.rand(1, T - n, qkv.shape[2], generator=gen) * 2 - 1) * 3e4).to(BF)
    mask = torch.ones(1, T)
    mask[:, n:] = 0
    alone = _run_bf16(qkv[:, :n].contiguous(), torch.ones(1, n), ek, ev, heads, cuda_device)
    padded = _run_bf16(qkv, mask, ek, ev, heads, cuda_device)
    assert torch.isfinite(padded.float()).all()
    assert torch.equal(alone, padded[:, :n])


@gpu
@pytest.mark.parametrize("T", [90, 385])
def test_attention_bf16_batch_invariant_and_deterministic(cuda_device, T):
    """Each utterance of a batch comes out identical to the same utterance run alone, and a second run is identical."""
    dk, heads, w = 16, 4, 4
    mask = _masks(T, T)
    qkv, ek, ev = _inputs(mask.shape[0], T, heads, dk, w, True, T)
    o = _run_bf16(qkv, mask, ek, ev, heads, cuda_device)
    assert torch.equal(o, _run_bf16(qkv, mask, ek, ev, heads, cuda_device))
    for b in range(mask.shape[0]):
        alone = _run_bf16(qkv[b:b + 1].contiguous(), mask[b:b + 1], ek, ev, heads, cuda_device)
        assert torch.equal(alone, o[b:b + 1])


@gpu
def test_attention_bf16_rejects_what_it_cannot_run(cuda_device):
    """w = 8 (the relative-key tile holds 16 rows) and T = 2049 (16 key tiles of key-mask words) are refused with
    VSG_EUNSUPPORTED (-4); so is dk = 128, whose tiles exceed a B200 block's shared memory (261 536 > 232 448 bytes).
    If dk = 128 runs on some device it must match the reference.  Never a raw CUDA error."""
    def refused(fn):
        with pytest.raises(RuntimeError) as e:
            fn()
        assert "failed (-4)" in str(e.value), str(e.value)
        return str(e.value)

    qkv, ek, ev = _inputs(1, 64, 2, 32, 8, False, 1)
    refused(lambda: _run_bf16(qkv, torch.ones(1, 64), ek, ev, 2, cuda_device))
    qkv, ek, ev = _inputs(1, 2049, 2, 32, 4, False, 2)
    refused(lambda: _run_bf16(qkv, torch.ones(1, 2049), ek, ev, 2, cuda_device))
    for heads in (1, 2):
        mask = _masks(200, heads)
        qkv, ek, ev = _inputs(mask.shape[0], 200, heads, 128, 4, True, 3)
        try:
            o = _heads(_run_bf16(qkv, mask, ek, ev, heads, cuda_device), heads, 128)
        except RuntimeError as e:
            assert "failed (-4)" in str(e) and "shared memory" in str(e), str(e)
            print(f"attention bf16 dk=128 h={heads}: {e}")
            continue
        _, ref_b = _references(qkv, mask, ek, ev, heads, 128, 4, cuda_device)
        assert float(_rel(o, ref_b).max()) <= TOL_B_MAX
    # the launcher still works after a refusal
    qkv, ek, ev = _inputs(1, 64, 2, 32, 4, False, 4)
    _run_bf16(qkv, torch.ones(1, 64), ek, ev, 2, cuda_device)


# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dk,heads,w,T", [(16, 4, 0, 1), (32, 2, 1, 63), (48, 4, 4, 65), (64, 2, 7, 129), (96, 2, 4, 1000),
                                          (128, 2, 4, 333), (128, 1, 8, 200), (64, 4, 4, 2048)])
def test_attention_f32_matches_fp64(cuda_device, dk, heads, w, T):
    """The fp32 kernel of the parity mode ([B, 3H, T] layout, online softmax over 64-key tiles) against (a) unrounded."""
    from visinger_b200 import _lib
    mask = _masks(T, T + w)
    for peaky in (True, False):
        qkv, ek, ev = _inputs(mask.shape[0], T, heads, dk, w, peaky, dk + T + w)
        qkv32 = qkv.float().transpose(1, 2).contiguous()
        o = _lib.debug_attention_f32(qkv32.to(cuda_device), mask, ek, ev, heads)
        o = _heads(o.transpose(1, 2), heads, dk)
        q, k, v = (t.to(cuda_device) for t in _split(qkv, heads, dk))
        ref = attention_fp64(q, k, v, mask.double().to(cuda_device), ek.double().to(cuda_device), ev.double().to(cuda_device), w)
        rel = _rel(o, ref)
        print(f"attention f32 dk={dk} h={heads} w={w} T={T} {'peaky' if peaky else 'flat'}: max {float(rel.max()):.2e}")
        assert float(rel.max()) <= TOL_F32_MAX


# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("C", [16, 32, 48, 96, 192, 256])
def test_layernorm_bf16_matches_fp64(cuda_device, C):
    """The bf16 encoder's fused LayerNorm -> + condition -> * mask step (relenc_layernorm_bf16_kernel) against float64
    from the same bf16 input, with no condition, a per-utterance and a per-frame one.  Rows with zero variance, rows with
    a large common offset (cancellation in the variance) and masked rows are part of every case."""
    from visinger_b200 import _lib
    B, T = 3, 77
    gen = torch.Generator().manual_seed(C)
    x = torch.randn(B, T, C, generator=gen) * 2
    x[:, 5] = 0.75                                                  # zero variance
    x[:, 6] = -3.0
    x[:, 7:12] = x[:, 7:12] + 300.0                                 # large mean, spread of a few bf16 ulps (2 at 300)
    x[:, 12:15] = x[:, 12:15] - 1000.0
    xb = x.to(BF)
    gamma = 1 + 0.1 * torch.randn(C, generator=gen)
    beta = 0.1 * torch.randn(C, generator=gen)
    mask = torch.ones(B, T)
    mask[1, 60:] = 0
    mask[2, ::9] = 0
    conds = [None, torch.randn(B, C, generator=gen), torch.randn(B, C, T, generator=gen)]
    for g in conds:
        y = _lib.debug_layernorm_bf16(xb.to(cuda_device), gamma, beta, mask, g).double().cpu()
        xd = xb.double()
        mu = xd.mean(-1, keepdim=True)
        var = (xd - mu).pow(2).mean(-1, keepdim=True)
        want = (xd - mu) / torch.sqrt(var + 1e-4) * gamma.double() + beta.double()
        if g is not None:
            want = want + (g.double()[:, None, :] if g.dim() == 2 else g.double().transpose(1, 2))
        want = want * mask.double()[..., None]
        # one bf16 ulp of each output (of 1/64 for outputs nearer 0, where fp32 cancellation against beta + g dominates)
        ulp = torch.exp2(torch.floor(torch.log2(want.abs().clamp_min(2 ** -6)))) / 128
        err = (y - want).abs()
        print(f"layernorm bf16 C={C} g={'none' if g is None else g.dim()}: max err {float((err / ulp).max()):.2f} ulp")
        assert float((err / ulp).max()) <= 1.0                     # measured 0.58 ulp
        assert float(y[mask == 0].abs().max()) == 0.0
