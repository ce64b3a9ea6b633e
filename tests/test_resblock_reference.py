"""The float64 references of the fused ResBlock1 kernels (tests/resblock_reference.py), on the CPU: they agree with an
independent fp32 emulation of each kernel that accumulates the second convolution the way the tensor pipe does
(truncating fp32, once per 16-wide K slice) in several orders, and the comparator rejects every fault a kernel rewrite
could make on the exact operands, by orders of magnitude over the gate."""
import pytest
import torch
import torch.nn.functional as F

import resblock_reference as R
from conv_reference import rel_err
from emulate_tc_accumulate import trunc32

ORDERS = ("tap", "chunk", "reverse")


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _bf(v):
    return v.float().to(torch.bfloat16).float()


def emulate(kind, xa, w1, b1, w2, b2, dil, *, add0=None, add0_is_act=False, add1=None, scale=1.0, order="tap"):
    """fp32 emulation of one live pair, written apart from the reference: conv1 by torch in fp32, the kernel's
    leaky_relu / rounding, conv2 as acc = trunc32(acc + one 16-channel tap slice) in the given order (rp: starting from the
    residual stream x0, which is that kernel's accumulator), then the epilogue's fp32 adds in the kernel's order."""
    s = torch.tensor(0.1, dtype=torch.float32)
    x = xa.float() if xa.dim() == 3 else xa[0].float() + xa[1].float()
    B, L, C = x.shape
    k = w1.shape[2]
    t = F.conv1d(x.transpose(1, 2), w1, b1, dilation=dil, padding=(k - 1) * dil // 2).transpose(1, 2)
    if kind == "rp":
        h = _bf(t)
        a = torch.where(h >= _bf(h * _bf(s)), h, _bf(h * _bf(s)))
    elif kind == "rp_x3":
        e = torch.where(t >= t * s, t, t * s)
        hi = _bf(e)
        a = hi.double() + _bf(e - hi).double()
    else:
        a = _bf(torch.where(t >= t * s, t, t * s))
    x0 = torch.where(x <= x * 10.0, x, x * 10.0)                 # fminf(f, f * 10.0f)
    acc = x0.clone() if kind in ("rp", "rp_x3") else torch.zeros(B, L, C)
    ap = F.pad(a.double(), (0, 0, (k - 1) // 2, (k - 1) // 2))
    slices = [(j, c0) for j in range(k) for c0 in range(0, C, 16)]
    if order == "chunk":
        slices.sort(key=lambda jc: (jc[1], jc[0]))
    elif order == "reverse":
        slices.reverse()
    for j, c0 in slices:
        part = ap[:, j:j + L, c0:c0 + 16] @ w2[:, c0:c0 + 16, j].double().T
        acc = trunc32(acc.double() + part)
    v = acc + b2
    if kind == "rb":
        v = v + x0
    if kind == "pair" and add0 is not None:
        r = add0.float()
        if add0_is_act:
            r = torch.where(r <= _bf(r * 10.0), r, _bf(r * 10.0))
        v = v + r
    if add1 is not None:
        v = v + (add1.float() if add1.dim() == 3 else add1[0].float() + add1[1].float())
    return v * scale if (scale != 1.0 or kind in ("rp", "rp_x3")) else v


def _case(kind, C, k, dil, B, L, seed, nonneg=False):
    g = _gen(seed)
    x3 = kind == "rp_x3"
    xa = R.exact_input(B, L, C, g, nonneg=nonneg, x3=x3)
    w1, b1 = R.exact_conv1(C, k, g)
    w2, b2 = R.dense_conv2(C, k, g)
    b1_alt = R.exact_conv1(C, k, g)[1]
    add1 = R.running_sum(B, L, C, g, x3=x3)
    kw = dict(add1=add1, scale=1.0 / 3.0)
    if kind == "pair":
        kw.update(add0=xa, add0_is_act=True)         # the decoder's form: the residual recovered from the activated input
    return xa, (w1, b1, w2, b2, dil), kw, b1_alt


CASES = [("pair", 16, 3, 1), ("pair", 32, 11, 5), ("rb", 16, 7, 3), ("rb", 64, 11, 5), ("rp", 16, 11, 5), ("rp", 32, 7, 3),
         ("rp_x3", 16, 7, 3), ("rp_x3", 32, 11, 5)]


@pytest.mark.parametrize("kind,C,k,dil", CASES)
def test_reference_agrees_with_truncating_fp32_emulation(kind, C, k, dil):
    """Every summation order of a truncating fp32 accumulator stays within the kernel's gate of the float64 reference,
    with and without the running sum and scale."""
    xa, conv, kw, _ = _case(kind, C, k, dil, 3, 300, C * 100 + k * 10 + dil)
    for extra in (kw, {k_: v for k_, v in kw.items() if k_ not in ("add1", "scale")}):
        want, S = R.reference(kind, xa, *conv, **extra)
        errs = [rel_err(emulate(kind, xa, *conv, order=o, **extra), want, S) for o in ORDERS]
        print(f"{kind} C={C} k={k} d={dil}: emulated floor {max(errs):.2e} (orders {', '.join(f'{e:.1e}' for e in errs)}), "
              f"gate {R.EPS[kind]:.1e}")
        assert max(errs) <= R.EPS[kind]


def _applies(kind, fault):
    if fault == "x3_drop_lo":
        return kind == "rp_x3"
    if fault in ("residual", "round_toward_zero", "ties_away"):
        # Two planes: the residual is recovered in fp32 from hi + lo, so there is no bf16 recovery to confuse it with.  A
        # wrong rounding mode in the split moves hi + lo by an ulp of the lo plane, 2^-16 of the intermediate: on these
        # operands that is 0.6 - 0.9x the gate, below what an fp32-accumulated conv2 can resolve.
        return kind != "rp_x3"
    return True


@pytest.mark.parametrize("kind,C,k,dil", CASES)
def test_comparator_rejects_each_fault(kind, C, k, dil):
    """The gate rejects each fault at some element, by a printed margin of at least 4x over the gate (at d = 1 the two
    dilation faults are the correct arithmetic and are skipped)."""
    xa, conv, kw, b1_alt = _case(kind, C, k, dil, 3, 300, C * 100 + k * 10 + dil + 1)
    got = emulate(kind, xa, *conv, **kw)
    lines = []
    for fault in R.FAULTS:
        if not _applies(kind, fault) or (dil == 1 and fault in ("conv2_dilated", "conv1_dil1")):
            continue
        want, S = R.reference(kind, xa, *conv, fault=fault, b1_alt=b1_alt, **kw)
        e = rel_err(got, want, S)
        n = int(((got.double() - want).abs() / S.clamp_min(2.0 ** -126) > R.EPS[kind]).sum())
        lines.append(f"  {fault:18s} rel {e:.2e} = {e / R.EPS[kind]:9.1f} x gate at {n} elements")
        assert e > 4 * R.EPS[kind], (fault, e)
    print(f"{kind} C={C} k={k} d={dil}:\n" + "\n".join(lines))


@pytest.mark.parametrize("kind", ("pair", "rb", "rp"))
def test_operands_exercise_the_rounding(kind):
    """The exact operands leave the intermediate's one bf16 rounding live: many values round inexactly and many are exact
    ties (where nearest-even and ties-away differ), at every channel count the kernel takes."""
    for C in ((16, 32, 64) if kind == "rb" else (16, 32)):
        g = _gen(C)
        xa = R.exact_input(1, 1024, C, g)
        w1, b1 = R.exact_conv1(C, 7, g)
        t = R.exact_t(R.input_value(xa), w1, b1, 3).float()
        s = torch.tensor(0.1, dtype=torch.float32)
        rounded = t if kind == "rp" else torch.maximum(t, t * s)     # what the kernel rounds to bf16 first
        inexact = float((rounded.to(torch.bfloat16).float() != rounded).float().mean())
        n_ties = R.ties(rounded)
        print(f"{kind} C={C}: {inexact:.0%} of {rounded.numel()} intermediates round inexactly, {n_ties} exact ties")
        assert inexact >= 0.3 and n_ties >= 500


@pytest.mark.parametrize("kind", ("rb", "rp", "rp_x3"))
def test_slot_construction(kind):
    """With xa >= 0 the re-activation after an all-zero slot gives the block input back (so slot q sees xa), and the
    exact-operand check refuses operands whose first convolution would round."""
    g = _gen(5)
    xa = R.exact_input(2, 200, 32, g, nonneg=True, x3=kind == "rp_x3")
    assert R.slot_input_check(kind, xa)
    ws, bs = R.slot_weights(32, 3, 3, 1, g)
    assert all(float(ws[i].abs().sum()) == 0 for i in (0, 1, 4, 5)) and float(bs[1].abs().sum()) == 0
    assert float(ws[2].abs().sum()) > 0 and float(bs[0].abs().sum()) > 0
    with pytest.raises(AssertionError):
        R.exact_t(R.input_value(xa) + 2.0 ** -20, ws[2], bs[2], 3)
