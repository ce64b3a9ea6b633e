"""Float64 statements of one launch of the convolution kernel (csrc/conv_tc.cuh), the bf16 roundings its epilogue
applies, and the comparators the epilogue tests gate with.

A launch computes, for utterance b, output row q < Lq (time step n = q * out_stride + out_phase) and channel co,
    acc[b, q, co] = sum_j sum_ci x[b, q + in_off0 + j * dil, ci] * w[co, ci, j]      (x = 0 outside 0 .. Lin - 1)
then its epilogue.  The references take the operands the kernel sees (bf16 values, or the sum of their bf16 planes) and
evaluate in float64; every gate is relative to S, the per-element sum of the magnitudes that enter the value (products,
bias, condition, adds), because fp32 accumulation error scales with S and not with the result."""
import torch
import torch.nn.functional as F

SLOPE = 0.1


def bf16(t):
    """Round to bf16 (nearest-even), returned in float64."""
    return t.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def planes(v, n):
    """Split fp32 values into n bf16 planes the way the kernel's epilogue does: hi = bf16(v), lo = bf16(v - hi), ..."""
    v = v.to(torch.float32)
    out = []
    for _ in range(n):
        h = v.to(torch.bfloat16)
        out.append(h)
        v = v - h.to(torch.float32)
    return out


def plane_value(ps):
    """Value carried by a list of bf16 planes, in float64."""
    return sum(p.to(torch.float64) for p in ps)


def operand(v, n):
    """The value the kernel sees for an fp32 operand carried in n bf16 planes."""
    return plane_value(planes(v, n))


def conv_ref(x, w, dil=1, in_off0=None, Lq=None, out_stride=1, out_phase=0):
    """acc and S_acc (sum of |products|) of one launch, float64.  x [B, Lin, Cin], w [Cout, Cin, k]; returns [B, Lq, Cout]
    over the output rows q (the caller places row q at time step q * out_stride + out_phase)."""
    x = x.to(torch.float64)
    w = w.to(torch.float64)
    B, Lin, Cin = x.shape
    Cout, _, k = w.shape
    if in_off0 is None:
        in_off0 = -((k - 1) * dil // 2)
    if Lq is None:
        Lq = Lin
    acc = torch.zeros(B, Lq, Cout, dtype=torch.float64)
    S = torch.zeros(B, Lq, Cout, dtype=torch.float64)
    q = torch.arange(Lq)
    for j in range(k):
        src = q + in_off0 + j * dil
        ok = (src >= 0) & (src < Lin)
        xs = torch.zeros(B, Lq, Cin, dtype=torch.float64)
        xs[:, ok] = x[:, src[ok]]
        acc += xs @ w[:, :, j].T
        S += xs.abs() @ w[:, :, j].abs().T
    return acc, S


def upsample_ref(x, w, bias, rate):
    """ConvTranspose1d(stride = rate, padding = (k - rate) / 2) in float64 (modules/visinger/decoder.py:46) and the sum of
    |products| + |bias|.  x [B, Lin, Cin], w [Cin, Cout, k]; returns [B, Lin * rate, Cout]."""
    k = w.shape[2]
    pad = (k - rate) // 2
    xt = x.to(torch.float64).transpose(1, 2)
    y = F.conv_transpose1d(xt, w.to(torch.float64), bias.to(torch.float64), stride=rate, padding=pad)
    S = F.conv_transpose1d(xt.abs(), w.to(torch.float64).abs(), bias.to(torch.float64).abs(), stride=rate, padding=pad)
    return y.transpose(1, 2), S.transpose(1, 2)


# ---- the epilogue's bf16 arithmetic, bit for bit -------------------------------------------------------------------

def act_bf16(v):
    """out_act of the one-plane epilogue from the fp32 value v: h = bf16(v), then max(h, bf16(h * bf16(slope))) on packed
    bf16 pairs (the product of two bf16 values is exact in fp32, so one rounding)."""
    h = v.to(torch.float32).to(torch.bfloat16).to(torch.float32)
    s = torch.tensor(SLOPE, dtype=torch.float32).to(torch.bfloat16).to(torch.float32)
    return torch.maximum(h, (h * s).to(torch.bfloat16).to(torch.float32)).to(torch.bfloat16)


def residual_from_act_bf16(a):
    """The one-plane epilogue's residual from an activated bf16 add: min(a, bf16(a * bf16(1 / slope))) (bf16(10) = 10)."""
    a = a.to(torch.float32)
    inv = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(SLOPE, dtype=torch.float32)
    s = inv.to(torch.bfloat16).to(torch.float32)
    return torch.minimum(a, (a * s).to(torch.bfloat16).to(torch.float32))


def act_planes(v, n=2):
    """out_act of the two- / three-plane epilogue: fmaxf(v, v * slope) in fp32, then split into planes."""
    v = v.to(torch.float32)
    return planes(torch.maximum(v, v * torch.tensor(SLOPE, dtype=torch.float32)), n)


def residual_from_act_planes(ps):
    """The two- / three-plane epilogue's residual: f = fp32 sum of the planes, fminf(f, f * fp32(1 / slope))."""
    f = ps[0].to(torch.float32)
    for p in ps[1:]:
        f = f + p.to(torch.float32)
    inv = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(SLOPE, dtype=torch.float32)
    return torch.minimum(f, f * inv)


# ---- comparators ----------------------------------------------------------------------------------------------------

def rel_err(got, want, S):
    """Worst |got - want| / S over the elements (S floored at the smallest normal fp32 so that exact zeros compare)."""
    d = (got.to(torch.float64) - want.to(torch.float64)).abs()
    return float((d / S.to(torch.float64).clamp_min(2.0 ** -126)).max()) if d.numel() else 0.0


def within(got, want, S, eps):
    return rel_err(got, want, S) <= eps


def bits_equal(a, b):
    """Same shape, dtype and bit patterns (so -0 differs from +0 and a NaN equals itself)."""
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    iv = {torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.float64: torch.int64}
    return torch.equal(a.contiguous().view(iv[a.dtype]), b.contiguous().view(iv[b.dtype]))
