"""The float64 references and bf16 emulations of tests/conv_reference.py, on the CPU: they agree with torch's own
convolutions and roundings, and the comparators the epilogue tests gate with reject the ways a kernel goes subtly wrong."""
import math

import pytest
import torch
import torch.nn.functional as F

import conv_reference as R

EPS = 8e-7          # the one-plane gate of test_gpu_conv_epilogues.py, relative to S
EPS_X3 = 4.5e-6     # its two-plane gate


def _gen(seed):
    return torch.Generator().manual_seed(seed)


@pytest.mark.parametrize("k,dil,L", [(1, 1, 5), (3, 1, 129), (7, 3, 64), (11, 5, 300)])
def test_conv_ref_matches_conv1d(k, dil, L):
    g = _gen(k * 10 + dil)
    x = torch.randn(2, L, 24, generator=g, dtype=torch.float64)
    w = torch.randn(16, 24, k, generator=g, dtype=torch.float64)
    acc, S = R.conv_ref(x, w, dil)
    want = F.conv1d(x.transpose(1, 2), w, dilation=dil, padding=(k - 1) * dil // 2).transpose(1, 2)
    assert torch.allclose(acc, want, rtol=0, atol=1e-12)
    assert torch.allclose(S, F.conv1d(x.abs().transpose(1, 2), w.abs(), dilation=dil, padding=(k - 1) * dil // 2)
                          .transpose(1, 2), rtol=0, atol=1e-12)


def test_conv_ref_offsets_and_phases():
    """Non-centred in_off0 and Lq rows: row q reads x[q + in_off0 + j * dil] (zero outside), as a shifted conv1d."""
    g = _gen(3)
    x = torch.randn(1, 40, 8, generator=g, dtype=torch.float64)
    w = torch.randn(4, 8, 3, generator=g, dtype=torch.float64)
    for in_off0 in (-4, -2, 0, 3):
        acc, _ = R.conv_ref(x, w, 2, in_off0, 30)
        xp = F.pad(x.transpose(1, 2), (64, 64))
        full = F.conv1d(xp, w, dilation=2).transpose(1, 2)    # full[t] reads xp[t + 2j] = x[t - 64 + 2j]
        assert torch.allclose(acc[0], full[0, 64 + in_off0:64 + in_off0 + 30], rtol=0, atol=1e-12)


@pytest.mark.parametrize("rate,k", [(5, 11), (3, 7), (2, 4), (4, 8)])
def test_upsample_ref_is_the_transposed_convolution(rate, k):
    """upsample_ref against the definition y[n] = sum_{i, j: i * rate + j - pad = n} x[i] w[j] + b, by direct summation."""
    g = _gen(rate + k)
    Cin, Cout, Lin = 6, 5, 9
    x = torch.randn(2, Lin, Cin, generator=g, dtype=torch.float64)
    w = torch.randn(Cin, Cout, k, generator=g, dtype=torch.float64)
    b = torch.randn(Cout, generator=g, dtype=torch.float64)
    y, S = R.upsample_ref(x, w, b, rate)
    pad = (k - rate) // 2
    want = b.expand(2, Lin * rate, Cout).clone()
    for i in range(Lin):
        for j in range(k):
            n = i * rate + j - pad
            if 0 <= n < Lin * rate:
                want[:, n] += x[:, i] @ w[:, :, j]
    assert y.shape == (2, Lin * rate, Cout)
    assert torch.allclose(y, want, rtol=0, atol=1e-12)
    assert bool((S >= y.abs() - 1e-12).all())


def test_plane_splits_match_torch_rounding():
    g = _gen(5)
    v = torch.randn(4096, generator=g) * torch.exp2(torch.randint(-20, 20, (4096,), generator=g).float())
    hi, lo = R.planes(v, 2)
    assert torch.equal(hi, v.to(torch.bfloat16))
    assert torch.equal(lo, (v - v.to(torch.bfloat16).float()).to(torch.bfloat16))
    # three planes carry an fp32 value exactly; two carry about 16 mantissa bits
    assert torch.equal(R.plane_value(R.planes(v, 3)), v.double())
    assert float(((R.plane_value([hi, lo]) - v.double()).abs() / v.double().abs()).max()) <= 2.0 ** -16
    assert torch.equal(R.bf16(v), v.to(torch.bfloat16).double())


def test_activation_emulations():
    """act = max(h, bf16(h * bf16(0.1))): the bf16(0.1) is not 0.1 (0x3DCD = 0.10009765625), and the product is rounded
    once; the residual min(a, bf16(a * 10)) returns a positive a unchanged."""
    g = _gen(6)
    v = torch.randn(1 << 16, generator=g)
    a = R.act_bf16(v)
    h = v.to(torch.bfloat16).float()
    assert torch.equal(a[v > 0], v[v > 0].to(torch.bfloat16))
    assert float(torch.tensor(0.1).to(torch.bfloat16)) == 0.10009765625
    assert torch.equal(a[v < 0].float(), (h[v < 0] * 0.10009765625).to(torch.bfloat16).float())
    r = R.residual_from_act_bf16(a)
    assert torch.equal(r[v > 0], a[v > 0].float())
    hp = R.act_planes(v, 2)
    f = hp[0].float() + hp[1].float()
    assert torch.equal(hp[0], torch.maximum(v, v * 0.1).to(torch.bfloat16))
    rr = R.residual_from_act_planes(hp)
    assert float((rr.double() - v.double()).abs().max()) <= 2.0 ** -14 * float(v.abs().max())
    assert torch.equal(rr[f > 0], f[f > 0])


def test_bits_equal():
    a = torch.tensor([0.0, 1.0])
    assert R.bits_equal(a, a.clone())
    assert not R.bits_equal(a, torch.tensor([-0.0, 1.0]))
    assert not R.bits_equal(a.to(torch.bfloat16), a)


# ---- the gates bite: each comparator rejects a perturbation of a correct result --------------------------------------

def _case(seed, B=2, L=300, C=64, k=7, planes=1):
    g = _gen(seed)
    x = torch.randn(B, L, C, generator=g)
    w = torch.randn(C, C, k, generator=g) / math.sqrt(C * k)
    b = 0.1 * torch.randn(C, generator=g)
    xs = R.planes(x, planes)
    ws = R.planes(w, planes)
    pairs = [(0, 0)] if planes == 1 else [(0, 0), (0, 1), (1, 0)]
    acc = S = 0
    for i, j in pairs:
        t, s = R.conv_ref(xs[i].double(), ws[j].double())
        acc, S = acc + t, S + s
    v = acc + b.double()
    S = S + b.double().abs()
    return v, S, b


def test_gate_rejects_a_dropped_bias_channel():
    v, S, b = _case(1)
    got = v.float()                                    # a correct kernel: fp32 rounding only
    assert R.within(got, v, S, EPS)
    bad = got.clone()
    bad[..., 37] -= b[37]
    assert not R.within(bad, v, S, EPS)


def test_gate_rejects_a_row_shifted_at_a_tile_border():
    v, S, _ = _case(2)
    got = v.float()
    bad = got.clone()
    bad[1, 128] = got[1, 127]
    assert not R.within(bad, v, S, EPS)


def test_gate_rejects_a_zeroed_lo_plane_chunk():
    """Two-plane output whose lo plane is lost in one 32-channel chunk: 2^-9 relative, far above the gate."""
    v, S, _ = _case(3, planes=2)
    hi, lo = R.planes(v.float(), 2)
    assert R.within(R.plane_value([hi, lo]), v, S, EPS_X3)
    lo_bad = lo.clone()
    lo_bad[..., 32:64] = 0
    assert not R.within(R.plane_value([hi, lo_bad]), v, S, EPS_X3)
    # a kernel that skipped the lo-plane products of the operands is caught by the fp32 comparator
    v1, S1, _ = _case(3, planes=1)
    assert not R.within(v1.float(), v, S, EPS_X3)


def test_emulation_rejects_slope_point_one():
    """act computed with slope 0.1 instead of bf16(0.1) differs in bits on some negative values."""
    g = _gen(4)
    v = torch.randn(1 << 14, generator=g)
    h = v.to(torch.bfloat16).float()
    wrong = torch.maximum(h, (h * 0.1).to(torch.bfloat16).float()).to(torch.bfloat16)
    assert not R.bits_equal(wrong, R.act_bf16(v))


def test_gate_rejects_a_wrong_coupling_sign_on_one_utterance():
    g = _gen(7)
    B, L, C = 3, 50, 32
    m = torch.randn(B, L, C, generator=g, dtype=torch.float64)
    x1 = torch.randn(B, L, C, generator=g, dtype=torch.float64)
    mask = torch.ones(B, L, 1, dtype=torch.float64)
    want = (x1 - m) * mask
    S = m.abs() + x1.abs()
    got = want.float()
    assert R.within(got, want, S, EPS)
    bad = got.clone()
    bad[1] = (m[1] + x1[1] * mask[1]).float()
    assert not R.within(bad, want, S, EPS)


def test_gate_rejects_a_mask_one_frame_late():
    v, S, _ = _case(8, B=2, L=100)
    lengths = [100, 61]
    mask = (torch.arange(100)[None, :] < torch.tensor(lengths)[:, None]).double()[..., None]
    want = v * mask
    late = (torch.arange(100)[None, :] < torch.tensor(lengths)[:, None] + 1).double()[..., None]
    assert R.within((v * mask).float(), want, S, EPS)
    assert not R.within((v * late).float(), want, S, EPS)
