"""Float64 statements of the fused ResBlock1 kernels (csrc/pair_tc.cuh, rb_tc.cuh, rp_tc.cuh) on operands for which their
arithmetic is exact up to the last convolution, each kernel's own bf16 roundings, and the faults the tests must catch.

A pair of ResBlock1 (decoder.py:91-104) is  x += conv2(leaky_relu(conv1_d(leaky_relu(x)) + b1)) + b2.  On the operands
built here the first convolution is exact in fp32 whatever the summation order or the tensor pipe's truncation:
  xa on a 2^-6 grid in [-2, 2] (one plane) or a 2^-10 grid (two planes, hi + lo), w1 on a 2^-6 grid in +-6/64, b1 on a
  2^-10 grid in [-1/2, 1/2]
so every partial sum of C k <= 704 products is a multiple of 2^-16 below 2^8 (24 bits).  The intermediate t = conv1 + b1 is
therefore known exactly, and so are its bf16 rounding (nearest-even, with real ties) and each kernel's leaky_relu.  Only the
second convolution's fp32 accumulation and the epilogue's fp32 adds remain, a few ulp of S, the per-element sum of the
magnitudes that enter the value (|products| + |bias| + |residual| + |running sum|, times |scale|).

The whole-resblock kernels are tested one pair slot q at a time: every other slot gets W1 = W2 = 0 and b2 = 0 (its b1 stays,
it meets only zero weights), so the slots before q leave x at x0 and the slots after q add exact zeros.  With xa >= 0 for
q > 0 the re-activation between slots is the identity, and slot q sees the block input itself, at its own dilation and its
own bias index.

W2 is rounded to bf16, so the lo weight plane of the split-bf16 (rp_x3) conv2 is zero here and the W_lo products are not
exercised; the dense-weight X3 tests of test_gpu_round2.py cover them at the fp32 tolerance.

The roundings, per kernel (slope = 0.1f as the launchers pass it):
  pair, rb   mid:  bf16(fmaxf(t, t * 0.1f))                          (pair_tc.cuh pair_mid_epilogue, rb_tc.cuh)
  rp         mid:  h = bf16(t); max(h, bf16(h * bf16(0.1)))           (rp_tc.cuh, bf16x2_scale_max on packed pairs)
  rp_x3      mid:  e = fmaxf(t, t * 0.1f); hi = bf16(e), lo = bf16(e - hi); conv2 sees hi + lo
  rb, rp     residual x0 = fminf(f, f * (1.0f / 0.1f)) in fp32 (x3: f = hi + lo)
  pair       residual = add0, or (add0_is_act) min(a, bf16(a * bf16(10))) of the conv epilogue (conv_tc.cuh)
  all        out = (x + bias sum + add1) * scale in fp32; raw = bf16(out); act per kernel:
             pair, rp: act_bf16(raw); rb: bf16(fmaxf(out, out * 0.1f)); rp_x3: the planes of fmaxf(out, out * 0.1f)
"""
import torch
import torch.nn.functional as F

from conv_reference import act_bf16, conv_ref, planes, residual_from_act_bf16

KERNELS = ("pair", "rb", "rp", "rp_x3")
SLOPE_F32 = torch.tensor(0.1, dtype=torch.float32)
SLOPE_BF16 = SLOPE_F32.to(torch.bfloat16).to(torch.float32)
INV_SLOPE_F32 = torch.tensor(1.0, dtype=torch.float32) / SLOPE_F32          # 1.0f / 0.1f = 10.0f

# gates on out_f32, relative to S at every element: about 2x the floors tests/test_gpu_resblock_exact.py measured on a
# B200 (1000 W power limit): pair 2.8e-7, rb 3.5e-7, rp 1.2e-6 at C <= 32 and 1.6e-6 at C = 64, rp_x3 2.2e-6.  rp_tc
# accumulates conv2 onto x itself (rp_tc.cuh: x += W2 * a in tensor memory), so each K slice truncates an ulp of |x0| (up
# to 10 |xa|), where rb_tc accumulates from zero and adds x in the epilogue; the CPU emulation of a truncating fp32
# accumulator (tests/test_resblock_reference.py) lands at the same floors.
EPS = {"pair": 6e-7, "rb": 8e-7, "rp": 3.2e-6, "rp_x3": 4.5e-6}

# faults a kernel rewrite could make; each must move out_f32 far above the fp32 floor somewhere
FAULTS = ("round_toward_zero", "ties_away", "slope", "residual", "other_leaky", "conv2_dilated", "conv1_dil1",
          "prev_bias", "row_shift", "add1_after_scale", "next_utterance", "x3_drop_lo")


# ---- roundings --------------------------------------------------------------------------------------------------------

def round_bf16(v, mode="nearest_even"):
    """fp32 -> bf16 values (as fp32): nearest-even (the kernels), or the faults toward zero / ties away from zero."""
    v = v.to(torch.float32).contiguous()
    if mode == "nearest_even":
        return v.to(torch.bfloat16).to(torch.float32)
    bits = v.view(torch.int32)
    trunc = (bits & ~0xFFFF).view(torch.float32)
    if mode == "toward_zero":
        return trunc
    assert mode == "away"
    up = ((bits & ~0xFFFF) + 0x10000).view(torch.float32)                  # next bf16 away from zero (same sign)
    return torch.where((bits & 0xFFFF) >= 0x8000, up, trunc)


def ties(v):
    """Number of fp32 values exactly halfway between two bf16 values (where nearest-even and away-from-zero differ or
    agree by the parity of the lower neighbour)."""
    return int(((v.to(torch.float32).contiguous().view(torch.int32) & 0xFFFF) == 0x8000).sum())


def mid_act(kind, t, mode="nearest_even", slope=None, other=False):
    """The activated intermediate conv2 reads, as float64, from the exact fp32 t = conv1 + b1."""
    t = t.to(torch.float32)
    packed = (kind == "rp") != other
    if kind == "rp_x3" and not other:
        s = SLOPE_F32 if slope is None else slope
        e = torch.maximum(t, t * s)
        hi = round_bf16(e, mode)
        lo = round_bf16(e - hi, mode)
        return hi.double() + lo.double(), hi.double()
    if packed:
        s = SLOPE_BF16 if slope is None else slope
        h = round_bf16(t, mode)
        return torch.maximum(h, round_bf16(h * s)).double(), None
    s = SLOPE_F32 if slope is None else slope
    return round_bf16(torch.maximum(t, t * s), mode).double(), None


def residual_fp32(f):
    """rb / rp: x0 = fminf(f, f * (1.0f / 0.1f)) in fp32."""
    f = f.to(torch.float32)
    return torch.minimum(f, f * INV_SLOPE_F32).double()


def out_act(kind, out_f32):
    """The kernel's out_act from its fp32 output: bf16 [.., C], or for rp_x3 the rows [hi (C) | lo (C)]."""
    v = out_f32.to(torch.float32)
    if kind in ("pair", "rp"):
        return act_bf16(v)
    e = torch.maximum(v, v * SLOPE_F32)
    if kind == "rb":
        return e.to(torch.bfloat16)
    return torch.cat(planes(e, 2), dim=-1)


def out_raw(kind, out_f32):
    """The kernel's out_raw: bf16(out) (rp_x3: the two planes [2][.., C])."""
    if kind == "rp_x3":
        return torch.stack(planes(out_f32, 2))
    return out_f32.to(torch.float32).to(torch.bfloat16)


# ---- operands ---------------------------------------------------------------------------------------------------------

def exact_input(B, L, C, gen, nonneg=False, x3=False):
    """The block input xa (bf16 planes) on the exact grid: one plane [B, L, C], or two planes [2][B, L, C]."""
    den = 1024 if x3 else 64
    v = torch.randint(0 if nonneg else -2 * den, 2 * den + 1, (B, L, C), generator=gen).double() / den
    if x3:
        return torch.stack(planes(v, 2))
    return v.to(torch.bfloat16)


def input_value(xa):
    """float64 value of a one- or two-plane input."""
    return xa.double() if xa.dim() == 3 else xa[0].double() + xa[1].double()


def exact_conv1(C, k, gen):
    w = torch.randint(-6, 7, (C, C, k), generator=gen).float() / 64
    b = torch.randint(-512, 513, (C,), generator=gen).float() / 1024
    return w, b


def dense_conv2(C, k, gen):
    w = (torch.randn(C, C, k, generator=gen) / (C * k) ** 0.5).to(torch.bfloat16).float()     # bf16 weights: W_lo = 0
    b = (torch.randn(C, generator=gen) * 0.1).float()
    return w, b


def running_sum(B, L, C, gen, x3=False):
    v = torch.randn(B, L, C, generator=gen)
    return torch.stack(planes(v, 2)) if x3 else v.to(torch.bfloat16)


def slot_weights(C, k, n_pairs, q, gen):
    """Weights [c1_0, c2_0, c1_1, ...] and biases of a resblock whose only live pair is slot q: every other slot has zero
    weights and b2 = 0 but its own exact b1 (which then meets only zero weights)."""
    ws, bs = [], []
    for p in range(n_pairs):
        w1, b1 = exact_conv1(C, k, gen)
        w2, b2 = dense_conv2(C, k, gen)
        if p != q:
            w1, w2, b2 = torch.zeros_like(w1), torch.zeros_like(w2), torch.zeros_like(b2)
        ws += [w1, w2]
        bs += [b1, b2]
    return ws, bs


def exact_t(xin, w1, b1, dil, flat=False):
    """t = conv1(xin) + b1, checked exact: float32 and float64 agree bit for bit.  xin float64 [B, L, C].  flat: the
    utterances as one sequence (the fault of reading the neighbour utterance instead of the zero padding)."""
    B, L, C = xin.shape
    if flat:
        xin = xin.reshape(1, B * L, C)
    k = w1.shape[2]
    pad = (k - 1) * dil // 2
    t64 = F.conv1d(xin.transpose(1, 2), w1.double(), b1.double(), dilation=dil, padding=pad).transpose(1, 2)
    t32 = F.conv1d(xin.float().transpose(1, 2), w1.float(), b1.float(), dilation=dil, padding=pad).transpose(1, 2)
    assert torch.equal(t64, t32.double()), "the first convolution is not exact in fp32 on these operands"
    return t64.reshape(B, L, C)


def _conv2(a, w2, dil, flat):
    B, L, C = a.shape
    y, S = conv_ref(a.reshape(1, B * L, C) if flat else a, w2, dil)
    return y.reshape(B, L, C), S.reshape(B, L, C)


# ---- the reference --------------------------------------------------------------------------------------------------

def reference(kind, xa, w1, b1, w2, b2, dil, *, add0=None, add0_is_act=False, add1=None, scale=1.0, fault=None,
              b1_alt=None):
    """float64 out and S of one live pair of `kind` on the exact input xa (the bf16 planes conv1 reads).  rb / rp / rp_x3:
    the residual is recovered from xa and b2 is the running bias sum at the slot; pair: add0 / add0_is_act.  add1: bf16 planes [B, L, C] or [2][B, L, C].  fault: one of FAULTS (b1_alt: the bias the prev_bias
    fault takes)."""
    assert kind in KERNELS and (fault is None or fault in FAULTS)
    flat = fault == "next_utterance"
    mode = {"round_toward_zero": "toward_zero", "ties_away": "away"}.get(fault, "nearest_even")
    xin = input_value(xa)
    t = exact_t(xin, w1, b1_alt if fault == "prev_bias" else b1, 1 if fault == "conv1_dil1" else dil, flat)
    slope = None
    if fault == "slope":      # the other slope constant: 0.1f in the packed leaky_relu, bf16(0.1) in the fp32 one
        slope = SLOPE_F32 if kind == "rp" else SLOPE_BF16
    a, hi = mid_act(kind, t, mode, slope, other=fault == "other_leaky")
    if fault == "x3_drop_lo":
        assert kind == "rp_x3"
        a = hi
    y, S = _conv2(a, w2, dil if fault == "conv2_dilated" else 1, flat)
    bias = b2.double().view(1, 1, -1)
    # the residual: the conv epilogue recovers it in bf16 (pair, add0_is_act), the whole-resblock kernels in fp32; the
    # fault swaps the two
    if kind == "pair" and not add0_is_act:
        assert fault != "residual"
        res = torch.zeros_like(y) if add0 is None else add0.double()
    elif (kind == "pair") != (fault == "residual"):
        assert kind != "rp_x3"
        res = residual_from_act_bf16(add0 if kind == "pair" else xa).double()
    else:
        res = residual_fp32(add0 if kind == "pair" else xin)
    x = y + bias + res
    S = S + bias.abs() + res.abs()
    if add1 is not None:
        s1 = input_value(add1)
        x = x * scale + s1 if fault == "add1_after_scale" else (x + s1) * scale
        S = (S + s1.abs()) * abs(scale)
    else:
        x, S = x * scale, S * abs(scale)
    if fault == "row_shift":
        x = x.clone()
        x[:, 128] = x[:, 127]
    return x, S


def slot_input_check(kind, xa):
    """The re-activation between slots of a resblock whose earlier slots are zero must give xa back (xa >= 0): the
    kernel's formula applied to x0 = residual(xa)."""
    x0 = residual_fp32(input_value(xa))
    if kind == "rp_x3":
        got = input_value(torch.stack(planes(torch.maximum(x0.float(), x0.float() * SLOPE_F32), 2)))
    elif kind == "rp":
        got = act_bf16(x0).double()
    else:
        got = torch.maximum(x0.float(), x0.float() * SLOPE_F32).to(torch.bfloat16).double()
    return torch.equal(got, input_value(xa))
