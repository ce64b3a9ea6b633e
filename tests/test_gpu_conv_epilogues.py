"""One launch of the convolution kernel (csrc/conv_tc.cuh) at a time, through vsg_debug_conv_tc and
vsg_debug_upsample_tc, against float64 on the operands the kernel sees (tests/conv_reference.py).

- Decoder epilogues: every specialised image (ACT, RES_ACT, LINEAR, SUM0, SUM1, FINAL and the _X3 twins) is launched
  with the EpiTC generator_forward_tc builds for it.  The generic image with an fp32 copy must match float64 within
  eps * S; its bf16 outputs must be the bit-exact roundings of that fp32 value; the specialised image (no fp32 copy)
  and the generic image (epi_sigs = 0) must give the same bits.
- Flow epilogues in the flow's layout (rows of planes * 2H, planes 2H apart): GATE with the speaker condition, in one
  plane (tanh.approx) and three planes (tanhf / expf); LINEAR with a mask; COUPLE in both signs.  Rows beyond each length
  are 0.
- Geometry: strided polyphase outputs leave the other rows untouched; non-centred input offsets; planar two-plane
  tensors give the bits of interleaved ones.
- The upsampler: merged and per-phase launches, one and two planes, planar and interleaved, against
  F.conv_transpose1d in float64, and bit-identical to each other.

Floors measured on a B200 (1000 W power limit), worst |got - want| / S over every case of the module; gates are about 2x:
  one plane (bf16 operands, fp32 accumulation)             3.9e-7 -> 8e-7
  two planes (three plane products per MAC)                2.1e-6 -> 4.5e-6
  three planes (six plane products per MAC)                1.3e-7 -> 3e-7
  GATE, one plane (tanh.approx): absolute error of the output 9.5e-6 -> 2e-5 (on top of the one-plane gate)
  upsampler, one and two planes                            1.6e-6 -> 3.2e-6
"""
import math

import pytest
import torch

import conv_reference as R

pytestmark = pytest.mark.gpu

EPS = {1: 8e-7, 2: 4.5e-6, 3: 3e-7}
GATE_FAST_ABS = 2e-5
UPS_EPS = 3.2e-6
SENTINEL = -768.0          # exact in bf16; no output of these tests can take it

_floors = {}


def _note(name, value):
    _floors[name] = max(_floors.get(name, 0.0), value)
    print(f"floor[{name}] so far {_floors[name]:.3e}")


def _lib():
    from visinger_b200 import _lib
    return _lib


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _plane_tensor(v, n):
    """fp32 values [.., C] -> bf16 tensor with rows [p0 | p1 | ..] (n planes) and the value the kernel sees."""
    ps = R.planes(v, n)
    return torch.cat(ps, -1).contiguous(), R.plane_value(ps)


def _split(t, n):
    C = t.shape[-1] // n
    return [t[..., i * C:(i + 1) * C] for i in range(n)]


def _products(x_ps, w_ps, dil, in_off0, Lq):
    """acc and S of the plane products the kernel issues: one plane a0 w0; two planes a0 w0 + a0 w1 + a1 w0; three planes
    the six products a2 w0, a1 w1, a1 w0, a0 w2, a0 w1, a0 w0."""
    n = len(x_ps)
    pairs = {1: [(0, 0)], 2: [(0, 0), (0, 1), (1, 0)], 3: [(2, 0), (1, 1), (1, 0), (0, 2), (0, 1), (0, 0)]}[n]
    acc = S = 0
    for a, b in pairs:
        t, s = R.conv_ref(x_ps[a].double(), w_ps[b].double(), dil, in_off0, Lq)
        acc = acc + t
        S = S + s
    return acc, S


# ---------------------------------------------------------------------------------------------------------------------
# decoder epilogues

# kind -> (add0 kind, add1, outputs, scale); add0 "act" = the activated running stream (add0_is_act), "raw" = a raw add
DECODER_KINDS = {
    "ACT": (None, False, ("act",), 1.0),
    "RES_ACT": ("act", False, ("act",), 1.0),
    "LINEAR": ("raw", False, ("raw", "act"), 1.0),        # the two-stream resblock (bit 12): raw and activated copies
    "SUM0": ("act", False, ("raw",), 1.0),
    "SUM1": ("act", True, ("raw",), 1.0),
    "FINAL": ("act", True, ("act",), 1.0 / 3.0),
}

# (C, k, dil, B, L): the decoder's channel widths, kernels and dilations; lengths on both sides of 128-row tile borders,
# and one launch with more tiles than 2 x 148 CTAs
DECODER_SHAPES = [
    (256, 3, 1, 1, 1), (256, 11, 5, 2, 129), (128, 7, 3, 3, 255), (128, 11, 1, 1, 1000), (64, 3, 5, 2, 127),
    (64, 7, 1, 1, 257), (32, 11, 3, 3, 128), (32, 3, 1, 2, 1000), (16, 7, 5, 1, 129), (16, 11, 1, 3, 255),
    (64, 3, 1, 3, 40000),
]


def _decoder_case(kind, planes, C, k, dil, B, L, seed, d):
    L_ = _lib()
    add0_kind, has_add1, outs, scale = DECODER_KINDS[kind]
    g = _gen(seed)
    x32 = torch.randn(B, L, C, generator=g)
    w = torch.randn(C, C, k, generator=g) / math.sqrt(C * k)
    bias = 0.1 * torch.randn(C, generator=g)
    x, _ = _plane_tensor(x32, planes)
    w_ps = R.planes(w, planes)
    acc, S = _products(_split(x, planes), w_ps, dil, None, L)
    v = acc + bias.double()
    S = S + bias.double().abs()
    args = dict(B=B, Lin=L, Lq=L, dil=dil, planes=planes, scale=scale)
    if add0_kind:
        a32 = torch.randn(B, L, C, generator=g)
        if add0_kind == "act":        # an activated stream, as the previous epilogue stored it
            a = torch.cat(R.act_planes(a32, planes), -1) if planes > 1 else R.act_bf16(a32)
            r = R.residual_from_act_planes(_split(a, planes)) if planes > 1 else R.residual_from_act_bf16(a)
            args.update(add0_is_act=1)
        else:
            a, _ = _plane_tensor(a32, planes)
            r = R.plane_value(_split(a, planes))
        v = v + r.double()
        S = S + r.double().abs()
        args["add0"] = a.to(d)
    if has_add1:
        a1, a1v = _plane_tensor(0.5 * torch.randn(B, L, C, generator=g), planes)
        v = v + a1v
        S = S + a1v.abs()
        args["add1"] = a1.to(d)
    v, S = v * scale, S * scale

    def outputs():
        return {o: torch.full((B, L, planes * C), SENTINEL, dtype=torch.bfloat16, device=d) for o in outs}

    # generic image with the fp32 copy
    og = outputs()
    f32 = torch.empty(B, L, C, dtype=torch.float32, device=d)
    img = L_.debug_conv_tc(x.to(d), w, bias, out_f32=f32, out_raw=og.get("raw"), out_act=og.get("act"), **args)
    assert img == L_.EPI_SIG["GENERIC"]
    f32 = f32.cpu()
    err = R.rel_err(f32, v, S)
    _note(f"planes{planes}", err)
    assert err <= EPS[planes], f"{kind} x{planes} C={C} k={k} d={dil} B={B} L={L}: {err:.3e} of S"
    # its bf16 outputs are the roundings of that fp32 value, bit for bit
    if "raw" in og:
        want = torch.cat(R.planes(f32, planes), -1)
        assert R.bits_equal(og["raw"].cpu(), want)
    if "act" in og:
        want = torch.cat(R.act_planes(f32, planes), -1) if planes > 1 else R.act_bf16(f32)
        assert R.bits_equal(og["act"].cpu(), want)
    # the specialised image, and the generic image without the fp32 copy: the same bits
    want_img = kind + ("_X3" if planes == 2 else "")
    for epi_sigs, name in ((2, want_img), (0, "GENERIC")):
        os_ = outputs()
        img = L_.debug_conv_tc(x.to(d), w, bias, out_raw=os_.get("raw"), out_act=os_.get("act"), epi_sigs=epi_sigs, **args)
        assert img == L_.EPI_SIG[name], f"{kind} x{planes} epi_sigs={epi_sigs}: launched image {img}"
        for o in outs:
            assert R.bits_equal(os_[o].cpu(), og[o].cpu()), f"{name} image differs from the generic one in {o}"


@pytest.mark.parametrize("C,k,dil,B,L", DECODER_SHAPES)
@pytest.mark.parametrize("kind", list(DECODER_KINDS))
def test_decoder_epilogue_one_plane(cuda_device, kind, C, k, dil, B, L):
    _decoder_case(kind, 1, C, k, dil, B, L, 1000 + C + k + L, cuda_device)


@pytest.mark.parametrize("C,k,dil,B,L", DECODER_SHAPES)
@pytest.mark.parametrize("kind", [k for k in DECODER_KINDS if k != "LINEAR"])
def test_decoder_epilogue_two_planes(cuda_device, kind, C, k, dil, B, L):
    """The bf16x3 decoder's images (ACT_X3 .. FINAL_X3): rows [hi | lo], three plane products per MAC."""
    _decoder_case(kind, 2, C, k, dil, B, L, 2000 + C + k + L, cuda_device)


# ---------------------------------------------------------------------------------------------------------------------
# flow epilogues (rows of planes * 2H channels, planes 2H apart, ragged lengths)

def _mask(lengths, L):
    return (torch.arange(L)[None, :] < torch.tensor(lengths)[:, None]).float()


def _flow_inputs(planes, H, Cin_ch, lengths, L, seed):
    g = _gen(seed)
    B = len(lengths)
    m = _mask(lengths, L)
    # hs: rows [h (H) | out (H)] per plane, the input of the gate conv is h (Cin_ch = H channels)
    h32 = torch.randn(B, L, H, generator=g) * m[..., None]
    hs = torch.zeros(B, L, planes * 2 * H, dtype=torch.bfloat16)
    hps = R.planes(h32, planes)
    for p in range(planes):
        hs[..., p * 2 * H:p * 2 * H + H] = hps[p]
    return g, m, hs, hps


@pytest.mark.parametrize("planes", [1, 3])
@pytest.mark.parametrize("H,k,dil,lengths,L", [(192, 5, 1, [100, 87, 1], 100), (64, 3, 2, [300, 129], 300),
                                               (192, 5, 1, [1000], 1000)])
def test_flow_gate_with_condition(cuda_device, planes, H, k, dil, lengths, L):
    """acts = tanh(a) * sigmoid(s) of in_layer(h) + bias + bcond (encoder.py:206-213), channel pairs (2c, 2c+1) = (a, s)."""
    L_ = _lib()
    d = cuda_device
    g, m, hs, hps = _flow_inputs(planes, H, H, lengths, L, 31 + H + planes)
    B = len(lengths)
    w = torch.randn(2 * H, H, k, generator=g) / math.sqrt(H * k)
    bias = 0.1 * torch.randn(2 * H, generator=g)
    NF = 3   # the condition table of several layers: bcond_bs floats between utterances, this layer's slice at an offset
    cond_all = 0.2 * torch.randn(B, NF * 2 * H, generator=g)
    off = 2 * H
    bcond = cond_all.to(d).reshape(-1)[off:]      # utterance b's slice starts at b * bcond_bs
    acc, S = _products(hps, R.planes(w, planes), dil, None, L)
    v = acc + bias.double() + cond_all[:, None, off:off + 2 * H].double()
    S = S + bias.double().abs() + cond_all[:, None, off:off + 2 * H].double().abs()
    want = torch.tanh(v[..., 0::2]) * torch.sigmoid(v[..., 1::2])
    f32 = torch.empty(B, L, H, dtype=torch.float32, device=d)
    raw = torch.full((B, L, planes * H), SENTINEL, dtype=torch.bfloat16, device=d)
    img = L_.debug_conv_tc(hs.to(d), w, bias, B=B, Lin=L, Lq=L, dil=dil, planes=planes, mode=L_.EPI_TC_GATE, bcond=bcond,
                           bcond_bs=NF * 2 * H, out_f32=f32, out_raw=raw, x_ld=planes * 2 * H, x_part_stride=2 * H)
    assert img == L_.EPI_SIG["X6" if planes == 3 else "GENERIC"]
    f32 = f32.cpu()
    # derivative of tanh(a) sigmoid(s) is at most 1 in each argument: the accumulation error passes through unamplified
    Sg = torch.maximum(S[..., 0::2], S[..., 1::2])
    d_ = (f32.double() - want).abs()
    if planes == 1:
        fast = float((d_ - EPS[1] * Sg).max())
        _note("gate_fast_abs", float(d_.max()))
        assert fast <= GATE_FAST_ABS
    else:
        err = float((d_ / (Sg + 1.0)).max())      # tanhf / expf: a few ulp of an O(1) result on top of the products
        _note("planes3", err)
        assert err <= EPS[3]
    assert R.bits_equal(raw.cpu(), torch.cat(R.planes(f32, planes), -1))



@pytest.mark.parametrize("planes", [1, 3])
@pytest.mark.parametrize("H,lengths,L", [(192, [100, 87, 1], 100), (64, [300, 129], 300)])
def test_flow_linear_with_mask(cuda_device, planes, H, lengths, L):
    """h = (h + res(acts) + bias) * mask written into the [h | out] rows (flow_forward_tc, un-merged): the `out` half is
    left untouched and rows beyond each length are exactly 0."""
    L_ = _lib()
    d = cuda_device
    g, m, hs, hps = _flow_inputs(planes, H, H, lengths, L, 77 + H + planes)
    B = len(lengths)
    acts32 = torch.randn(B, L, H, generator=g)
    acts, _ = _plane_tensor(acts32, planes)
    w = torch.randn(H, H, 1, generator=g) / math.sqrt(H)
    bias = 0.1 * torch.randn(H, generator=g)
    acc, S = _products(_split(acts, planes), R.planes(w, planes), 1, 0, L)
    hv = R.plane_value(hps)
    v = (acc + bias.double() + hv) * m[..., None].double()
    S = S + bias.double().abs() + hv.abs()
    out = hs.clone()
    for p in range(planes):
        out[..., p * 2 * H + H:(p + 1) * 2 * H] = SENTINEL
    out = out.to(d)
    f32 = torch.empty(B, L, H, dtype=torch.float32, device=d)
    img = L_.debug_conv_tc(acts.to(d), w, bias, B=B, Lin=L, Lq=L, planes=planes, mask=m.to(d).contiguous(), add0=out,
                           out_raw=out, out_f32=f32, ld=planes * 2 * H, part_stride=2 * H)
    assert img == L_.EPI_SIG["X6" if planes == 3 else "GENERIC"]
    f32, out = f32.cpu(), out.cpu()
    err = R.rel_err(f32, v, S)
    _note(f"planes{planes}", err)
    assert err <= EPS[planes]
    for b, n in enumerate(lengths):
        assert bool((f32[b, n:] == 0).all())
    got = torch.cat([out[..., p * 2 * H:p * 2 * H + H] for p in range(planes)], -1)
    assert R.bits_equal(got, torch.cat(R.planes(f32, planes), -1))
    for p in range(planes):
        assert bool((out[..., p * 2 * H + H:(p + 1) * 2 * H].float() == SENTINEL).all())


@pytest.mark.parametrize("planes", [1, 3])
@pytest.mark.parametrize("sign", [-1, 1])
def test_flow_coupling(cuda_device, planes, sign):
    """m = (post(out) + bias) * mask; x1 = (x1 - m) * mask (reverse) | m + x1 * mask (forward), flow.py:78,83, in place on
    the half of the coupling state u that the step updates; the other half is untouched."""
    L_ = _lib()
    d = cuda_device
    H, C, lengths, L = 192, 192, [130, 128, 5], 130
    half = C // 2
    g, m, hs, hps = _flow_inputs(planes, H, H, lengths, L, 5 + planes + sign)
    B = len(lengths)
    for p in range(planes):        # the skip sum `out` is the input here
        hs[..., p * 2 * H + H:(p + 1) * 2 * H] = hs[..., p * 2 * H:p * 2 * H + H]
    outp = [hps[p] for p in range(planes)]
    w = torch.randn(half, H, 1, generator=g) / math.sqrt(H)
    bias = 0.1 * torch.randn(half, generator=g)
    u32 = torch.randn(B, L, C, generator=g)
    ups = R.planes(u32, planes)
    u = torch.cat(ups, -1).contiguous()
    x1v = R.plane_value([p[..., half:] for p in ups])
    acc, S = _products(outp, R.planes(w, planes), 1, 0, L)
    mm = m[..., None].double()
    mv = (acc + bias.double()) * mm
    want = (x1v - mv) * mm if sign < 0 else mv + x1v * mm
    S = (S + bias.double().abs()) + x1v.abs()
    ud = u.to(d)
    x1 = ud.reshape(-1)[half:]           # x1 = u + half: rows of planes * C, planes C apart
    f32 = torch.empty(B, L, half, dtype=torch.float32, device=d)
    img = L_.debug_conv_tc(hs.to(d).reshape(-1)[H:], w, bias, B=B, Lin=L, Lq=L,
                           planes=planes, mode=L_.EPI_TC_COUPLE, couple_sign=sign, mask=m.to(d).contiguous(), add0=x1,
                           out_raw=x1, out_f32=f32, ld=planes * C, part_stride=C, x_ld=planes * 2 * H, x_part_stride=2 * H)
    assert img == L_.EPI_SIG["X6" if planes == 3 else "GENERIC"]
    f32, uo = f32.cpu(), ud.cpu()
    err = R.rel_err(f32, want, S)
    _note(f"planes{planes}", err)
    assert err <= EPS[planes]
    for b, n in enumerate(lengths):
        assert bool((f32[b, n:] == 0).all())
    got = torch.cat([uo[..., p * C + half:(p + 1) * C] for p in range(planes)], -1)
    assert R.bits_equal(got, torch.cat(R.planes(f32, planes), -1))
    for p in range(planes):
        assert R.bits_equal(uo[..., p * C:p * C + half], u[..., p * C:p * C + half])


# ---------------------------------------------------------------------------------------------------------------------
# output geometry

@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("rate,k,Lin", [(5, 3, 100), (2, 2, 129), (3, 3, 1)])
def test_strided_phase_outputs(cuda_device, planes, rate, k, Lin):
    """Phase r of a polyphase output writes time steps q * rate + r only: every other row keeps its sentinel."""
    L_ = _lib()
    d = cuda_device
    B, C = 2, 64
    g = _gen(rate * 100 + k + planes)
    x, _ = _plane_tensor(torch.randn(B, Lin, C, generator=g), planes)
    w = torch.randn(C, C, k, generator=g) / math.sqrt(C * k)
    bias = 0.1 * torch.randn(C, generator=g)
    Lout = Lin * rate
    act = torch.full((B, Lout, planes * C), SENTINEL, dtype=torch.bfloat16, device=d)
    written = torch.zeros(Lout, dtype=torch.bool)
    for r in range(rate):
        Lq = (Lout - r + rate - 1) // rate
        in_off0 = -(k - 1) + (r % 2)             # not centred
        f32 = torch.empty(B, Lout, C, dtype=torch.float32, device=d)
        act_r = torch.full_like(act, SENTINEL)
        img = L_.debug_conv_tc(x.to(d), w, bias, B=B, Lin=Lin, Lq=Lq, Lout=Lout, in_off0=in_off0, out_stride=rate, out_phase=r,
                               planes=planes, out_act=act_r, out_f32=f32)
        assert img == L_.EPI_SIG["GENERIC"]
        acc, S = _products(_split(x, planes), R.planes(w, planes), 1, in_off0, Lq)
        rows = torch.arange(Lq) * rate + r
        f32 = f32.cpu()[:, rows]
        err = R.rel_err(f32, acc + bias.double(), S + bias.double().abs())
        _note(f"planes{planes}", err)
        assert err <= EPS[planes]
        act_r = act_r.cpu()
        want = torch.cat(R.act_planes(f32, planes), -1) if planes > 1 else R.act_bf16(f32)
        assert R.bits_equal(act_r[:, rows], want)
        others = torch.ones(Lout, dtype=torch.bool)
        others[rows] = False
        assert bool((act_r[:, others].float() == SENTINEL).all())
        # the production image (ACT / ACT_X3) writes the same rows with the same bits
        act_s = torch.full_like(act, SENTINEL)
        img = L_.debug_conv_tc(x.to(d), w, bias, B=B, Lin=Lin, Lq=Lq, Lout=Lout, in_off0=in_off0, out_stride=rate, out_phase=r,
                               planes=planes, out_act=act_s)
        assert img == L_.EPI_SIG["ACT_X3" if planes == 2 else "ACT"]
        assert R.bits_equal(act_s.cpu(), act_r)
        written[rows] = True
    assert bool(written.all())


@pytest.mark.parametrize("C,k,dil,B,L", [(64, 7, 3, 2, 300), (32, 3, 1, 3, 129), (128, 11, 5, 1, 257)])
def test_planar_equals_interleaved(cuda_device, C, k, dil, B, L):
    """Two-plane tensors as whole planes (ld = C, planes B * L * C apart) give the bits of rows [hi | lo], for the input,
    the adds and both outputs."""
    L_ = _lib()
    d = cuda_device
    g = _gen(C + k + L)
    x, _ = _plane_tensor(torch.randn(B, L, C, generator=g), 2)
    a0 = torch.cat(R.act_planes(torch.randn(B, L, C, generator=g), 2), -1)
    a1, _ = _plane_tensor(torch.randn(B, L, C, generator=g), 2)
    w = torch.randn(C, C, k, generator=g) / math.sqrt(C * k)
    bias = 0.1 * torch.randn(C, generator=g)

    def planar(t):
        return torch.stack(_split(t, 2)).contiguous()

    for outs in (("raw",), ("act",), ("raw", "act")):
        kw = dict(B=B, Lin=L, Lq=L, dil=dil, planes=2, add0=a0.to(d), add0_is_act=1, add1=a1.to(d), scale=0.5)
        o_i = {o: torch.full((B, L, 2 * C), SENTINEL, dtype=torch.bfloat16, device=d) for o in outs}
        L_.debug_conv_tc(x.to(d), w, bias, out_raw=o_i.get("raw"), out_act=o_i.get("act"), **kw)
        kw.update(add0=planar(a0).to(d), add1=planar(a1).to(d))
        o_p = {o: torch.full((2, B, L, C), SENTINEL, dtype=torch.bfloat16, device=d) for o in outs}
        L_.debug_conv_tc(planar(x).to(d), w, bias, out_raw=o_p.get("raw"), out_act=o_p.get("act"), x_ld=C,
                         x_part_stride=B * L * C, ld=C, part_stride=B * L * C, **kw)
        for o in outs:
            assert R.bits_equal(o_p[o].cpu(), planar(o_i[o].cpu())), f"planar {o} differs"


# ---------------------------------------------------------------------------------------------------------------------
# the upsampler (ConvTranspose1d as per-phase or merged convolutions, pack_upsampler / launch_upsample_tc)

# (rate, k, Cin, Cout): every stage of VISINGER_GENERATOR and of the ResBlock2 test configuration
UPSAMPLERS = [(5, 11, 512, 256), (5, 11, 256, 128), (3, 7, 128, 64), (2, 4, 64, 32), (2, 4, 32, 16),
              (4, 8, 128, 64), (2, 4, 64, 32)]


@pytest.mark.parametrize("rate,k,Cin,Cout", UPSAMPLERS)
@pytest.mark.parametrize("planes", [1, 2])
def test_upsampler_vs_conv_transpose(cuda_device, rate, k, Cin, Cout, planes):
    L_ = _lib()
    d = cuda_device
    B, lengths = 2, (1, 37, 130)
    g = _gen(rate * 1000 + k * 10 + Cin + planes)
    w = torch.randn(Cin, Cout, k, generator=g) / math.sqrt(Cin * k / rate)
    bias = 0.1 * torch.randn(Cout, generator=g)
    w_ps = R.planes(w, planes)
    for Lin in lengths:
        x, _ = _plane_tensor(torch.randn(B, Lin, Cin, generator=g), planes)
        x_ps = _split(x, planes)
        pairs = [(0, 0)] if planes == 1 else [(0, 0), (0, 1), (1, 0)]
        want = S = 0
        for a, b in pairs:
            y, s = R.upsample_ref(x_ps[a].double(), w_ps[b].double(), torch.zeros(Cout), rate)
            want, S = want + y, S + s
        want, S = want + bias.double(), S + bias.double().abs()
        Lout = Lin * rate
        layouts = [(0, False, False)] if planes == 1 else [(2, False, False), (2 | 4, True, False), (2 | 8, False, True),
                                                             (2 | 4 | 8, True, True)]
        results = {}
        for flags, pin, pout in layouts:
            xin = torch.stack(x_ps).contiguous() if pin else x
            for merged in (0, 1):
                if merged and planes == 2 and not pout:
                    continue                       # the two-plane merged form writes planar planes only
                fl = flags | merged
                shape = (planes, B, Lout, Cout) if pout else (B, Lout, planes * Cout)
                act = torch.full(shape, SENTINEL, dtype=torch.bfloat16, device=d)
                raw = torch.full(shape, SENTINEL, dtype=torch.bfloat16, device=d)
                f32 = torch.empty(B, Lout, Cout, dtype=torch.float32, device=d)
                img = L_.debug_upsample_tc(xin.to(d), w, bias, rate, fl, act, raw, f32)
                assert img == L_.EPI_SIG["GENERIC"]
                act_p = torch.full(shape, SENTINEL, dtype=torch.bfloat16, device=d)
                img = L_.debug_upsample_tc(xin.to(d), w, bias, rate, fl, act_p)      # what the decoder runs
                assert img == L_.EPI_SIG["ACT_X3" if planes == 2 else "ACT"]
                f32, act, raw, act_p = f32.cpu(), act.cpu(), raw.cpu(), act_p.cpu()
                assert R.bits_equal(act_p, act)
                if pout:
                    act, raw = torch.cat(list(act), -1), torch.cat(list(raw), -1)
                err = R.rel_err(f32, want, S)
                _note("upsampler", err)
                assert err <= UPS_EPS, f"rate {rate} k {k} {Cin}->{Cout} x{planes} flags {fl} Lin {Lin}: {err:.3e} of S"
                assert R.bits_equal(raw, torch.cat(R.planes(f32, planes), -1))
                want_act = torch.cat(R.act_planes(f32, planes), -1) if planes > 1 else R.act_bf16(f32)
                assert R.bits_equal(act, want_act)
                results[(pin, pout, merged)] = (f32, act)
        # merged and per-phase launches are the same sums in the same K order (the merged fold only adds zero taps)
        for (pin, pout, merged), (f32, act) in results.items():
            ref_f32, ref_act = results[(False, pout, 0)] if (False, pout, 0) in results else results[(pin, pout, 0)]
            assert R.bits_equal(f32, ref_f32) and R.bits_equal(act, ref_act), f"layout {(pin, pout, merged)} differs"
