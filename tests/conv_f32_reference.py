"""Float64 statements of one launch of the fp32 FFMA kernels (csrc/kernels_f32.cuh): the convolution with each fused
epilogue, the upsampler's polyphase launches, conv_post and the condition GEMV; the operands the tests feed them, the
gates, the GPU case matrix and the faults the gates must reject.

One launch of conv_f32_kernel, for utterance b, output row q < Lq (time step n = q * out_stride + out_phase < Lout) and
output channel co (layout [B, C, T], time contiguous; see vsg_debug_conv_f32 in include/visinger_b200.h):
    v[co] = sum_{ci, j} w[co, ci, j] * f(x[b, ci, q + in_off0 + j * dil]) + bias[co] + bcond[b, co]
x is zero outside [0, Lin) and f = leaky_relu(., slope) on load when asked, in fp32 as the kernel does it (so the operand
the products see is known exactly).  Then the epilogue, as the reference modules state it:
    LINEAR    u = (v + res) * mask;  y = u | y + u | (y + u) / NK              (decoder.py:48-54,102, rel_transformer.py)
    GATE      y[c] = tanh(v[c]) * sigmoid(v[c + H])  (the gate-interleaved pack)  (encoder.py:206-213)
    RES_SKIP  co < rs_split: h = (h + v) * mask;  else skip = v | skip + v, * mask on the last layer  (encoder.py:188-195)
    COUPLE    m = v * mask;  x1 = (x1 - m) * mask (reverse) | m + x1 * mask (forward)   (flow.py:70,78,83)
    MAG       y[c] = sqrt(v[2c]^2 + v[2c + 1]^2 + 1e-6) * mask, no bias            (spec.cuh)

Two operand layers:

* Exact operands (the method of tests/resblock_reference.py): x on a 2^-6 grid in [-2, 2], w on a 2^-6 grid in +-4/64,
  bias / bcond / res / the old y, y2 and x1 on a 2^-15 grid, load slopes 0 or 1/8.  Every product is then a multiple of
  2^-15 and so is every partial sum; a sum stays exact in fp32, in any order, while |sum| < 2^24 * 2^-15 = 512.
  `exact_bound` states the worst partial sum of a case and every case of the GPU matrix is checked against it.  On these
  operands LINEAR, RES_SKIP, COUPLE and ADD are known exactly; ADD_DIV is one IEEE division of an exact fp32 value, so
  torch's fp32 `/` gives its bits; GATE, MAG and conv_post's tanh are within the documented ulp bounds of tanhf (2 ulp),
  expf (2 ulp) and sqrtf (correctly rounded) plus their explicit roundings (the build does not use --use_fast_math).
  A missing tap, channel or term of any size shows.  (The upsampler's load slope is the production 0.1, so its exact
  operands are x >= 0.)
* Random operands at realistic magnitudes with the production slope 0.1.  The gate is the provable bound of an fp32 FMA
  chain, gamma_{n+m} * S with gamma_j = j u / (1 - j u), u = 2^-24, n = Cin * k products and m the epilogue's roundings,
  S the per-element sum of |products| + |bias| + |bcond| + |res| + |old value|.  GATE propagates it through |tanh'| <= 1
  and |sigmoid'| <= 1/4.  This layer catches precision loss: bf16 or TF32 operands.

Each named fault (FAULTS) is applied to the reference itself; tests/test_conv_f32_reference.py shows that the gate of the
layer that targets it rejects it.
"""
import math

import torch
import torch.nn.functional as F

U = 2.0 ** -24
GRID_X, GRID_W, GRID_ADD = 2.0 ** -6, 2.0 ** -6, 2.0 ** -15
X_MAX, W_MAX = 2.0, 4.0 / 64
BIAS_MAX, BCOND_MAX, RES_MAX, OLD_MAX = 1.0, 1.0, 2.0, 4.0
EXACT_SLOPE = 0.125
SLOPE = 0.1
MAG_EPS = float(torch.tensor(1e-6, dtype=torch.float32))
TINY = 2.0 ** -126
CI_CHUNK = 8                       # F32_CI_CHUNK: input channels staged per pass

LINEAR, GATE, RES_SKIP, COUPLE, MAG = 0, 1, 2, 3, 4
ACC_SET, ACC_ADD, ACC_ADD_DIV = 0, 1, 2

# fault -> the layers whose gate must reject it
FAULTS = {
    "tail_chunk": ("exact", "random"),        # the Cin % 8 tail chunk dropped
    "last_tap": ("exact", "random"),          # the last tap dropped
    "in_off0": ("exact", "random"),           # in_off0 off by one
    "right_clamp": ("exact", "random"),       # right-edge padding clamped to x[Lin - 1] instead of zeroed
    "mask_bs_lout": ("exact", "random"),      # mask row stride taken as Lout
    "bcond_neighbour": ("exact", "random"),   # bcond of the neighbouring utterance
    "gate_swap": ("exact", "random"),         # gate halves swapped
    "bias_twice": ("exact", "random"),
    "y2_first_ignored": ("exact", "random"),  # the first layer's skip sum accumulated onto stale memory
    "skip_mask_missing": ("exact", "random"), # the last layer's skip sum not masked
    "rs_split_8": ("exact", "random"),        # rs_split off by 8
    "couple_sign": ("exact", "random"),
    "x1_from_y": ("exact", "random"),         # COUPLE's x1 read from y instead of res
    "add_div_mul": ("exact",),                # ADD_DIV as a multiply by fp32(1 / NK) (NK = 3)
    "mag_no_eps": ("exact", "random"),        # MAG without the 1e-6
    "phase_off": ("exact", "random"),         # strided output phase off by one
    "ups_taps_reversed": ("exact", "random"), # one upsampler phase's taps reversed
    "post_ignores_n0": ("exact", "random"),   # conv_post computes samples [0, n1 - n0) instead of [n0, n1)
    "bf16": ("random",),                      # operands rounded to bf16
    "tf32": ("random",),                      # operands rounded to TF32
}


def gamma(j):
    return j * U / (1.0 - j * U)


# ---- the case matrix ---------------------------------------------------------------------------------------------------

def case(name, **kw):
    """One launch of the fp32 convolution.  Defaults: B = 3, centred taps, a dense output of Lq = Lin rows, LINEAR, bias,
    padded rows and guard channels in every buffer."""
    c = dict(name=name, B=3, Cin=8, Cout=16, k=1, dil=1, Lin=64, Lq=None, in_off0=None, out_stride=1, out_phase=0,
             Lout=None, epi=LINEAR, pre_lrelu=0, relu=False, bias=True, bcond=False, res="none", mask=False,
             acc_mode=ACC_SET, nk=1, rs_split=0, y2_first=0, y2_mask=0, couple_sign=1, gate_interleave=0,
             zero_frames=False, seed=0)
    c.update(kw)
    if c["in_off0"] is None:
        c["in_off0"] = -((c["k"] - 1) * c["dil"] // 2)
    if c["Lq"] is None:
        c["Lq"] = c["Lin"]
    if c["Lout"] is None:
        c["Lout"] = (c["Lq"] - 1) * c["out_stride"] + c["out_phase"] + 1
    if not c["seed"]:
        c["seed"] = 1 + sum(ord(ch) * (i + 1) for i, ch in enumerate(name)) % 100003
    return c


def ychannels(c):
    return {GATE: c["Cout"] // 2, MAG: c["Cout"] // 2, RES_SKIP: c["rs_split"]}.get(c["epi"], c["Cout"])


def exact_bound(n_products, adds):
    """Worst |partial sum| on the exact operands in units of the common grid 2^-15, for n_products products of at most
    W_MAX * X_MAX and additive terms of at most `adds` in all: the sums are exact in fp32 when this is below 2^24."""
    return (n_products * W_MAX * X_MAX + adds) / GRID_ADD


def conv_exact_bound(c):
    return exact_bound(c["Cin"] * c["k"], BIAS_MAX + BCOND_MAX + RES_MAX + OLD_MAX)


def _plan_q(Cout):
    return 1024 if Cout <= 16 else 512 if Cout <= 32 else 256


def gpu_cases():
    """The launches tests/test_gpu_conv_f32.py runs (each on both operand layers)."""
    cs = []
    # tile configurations: Cout around each switch, Lq around each configuration's Q, Cin around the 8-channel chunk
    for Cout in (1, 2, 15, 16, 17, 32, 33, 64, 65, 192, 576):
        Q = _plan_q(Cout)
        for Lq in (1, Q - 1, Q, Q + 1, 3 * Q + 5):
            if Cout >= 192 and Lq not in (Q + 1, 3 * Q + 5):
                continue
            cs.append(case(f"tile-co{Cout}-lq{Lq}", Cout=Cout, Cin=9, k=3, Lin=Lq, Lq=Lq))
    for Cin in (1, 7, 8, 9, 192, 513):
        cs.append(case(f"cin{Cin}", Cin=Cin, Cout=33, k=3, Lin=300))
    # taps at the shipped shapes, and a flow with dilation_rate 2 (5 taps at dilation 16)
    for k, dil, Cin, Cout in ((1, 1, 96, 192), (5, 1, 192, 384), (7, 1, 192, 512), (3, 1, 256, 256), (3, 3, 64, 64),
                              (3, 5, 32, 32), (7, 1, 128, 128), (7, 3, 64, 64), (7, 5, 16, 16), (11, 1, 256, 256),
                              (11, 3, 32, 32), (11, 5, 16, 16), (9, 1, 192, 768), (5, 16, 192, 384)):
        cs.append(case(f"taps-k{k}-d{dil}-{Cin}x{Cout}", Cin=Cin, Cout=Cout, k=k, dil=dil, Lin=271, pre_lrelu=1))
    # shared memory: the largest window under 48 KB and the smallest over it (k = 2, Cout > 32: 32 (384 + dil) bytes)
    cs.append(case("smem-48k-under", Cin=9, Cout=40, k=2, dil=1152, Lin=1300))
    cs.append(case("smem-48k-over", Cin=9, Cout=40, k=2, dil=1153, Lin=1300))
    cs.append(case("smem-200k-under", Cin=9, Cout=40, k=5, dil=1456, Lin=6000, Lq=300, in_off0=-2900))
    # LINEAR: +-bias, +-bcond, res separate and res == y, masks, SET / ADD / ADD_DIV at NK = 2 and 3, ReLU on load
    for bias in (False, True):
        for bcond in (False, True):
            cs.append(case(f"lin-b{int(bias)}-c{int(bcond)}", Cin=9, Cout=33, k=5, Lin=300, bias=bias, bcond=bcond,
                           mask=True))
    for res in ("sep", "alias"):
        for acc, nk in ((ACC_SET, 1), (ACC_ADD, 2), (ACC_ADD_DIV, 2), (ACC_ADD_DIV, 3)):
            cs.append(case(f"lin-res{res}-acc{acc}-nk{nk}", Cin=16, Cout=16, k=3, dil=3, Lin=300, res=res, acc_mode=acc,
                           nk=nk, pre_lrelu=1))
    cs.append(case("lin-relu", Cin=40, Cout=24, k=1, Lin=300, pre_lrelu=1, relu=True, res="alias"))
    cs.append(case("lin-ffn1-mask", Cin=24, Cout=40, k=9, Lin=300, mask=True))
    # GATE with the speaker condition (bcond_bs > Cout), interleaved as the flow / encoder pack it, and pre-interleaved
    for Cout, k, dil in ((32, 5, 1), (384, 5, 2), (96, 5, 16)):
        cs.append(case(f"gate-{Cout}-k{k}-d{dil}", Cin=Cout // 2, Cout=Cout, k=k, dil=dil, Lin=300, epi=GATE,
                       bcond=True, gate_interleave=1))
    cs.append(case("gate-packed-order", Cin=9, Cout=18, k=3, Lin=300, epi=GATE, bcond=True))
    # RES_SKIP: rs_split = H (a middle layer) and 0 (the last layer) x y2_first x y2_mask
    for rs in (1, 0):
        for first in (0, 1):
            for ymask in (0, 1):
                H = 48
                cs.append(case(f"rs-split{rs}-first{first}-mask{ymask}", Cin=H, Cout=2 * H if rs else H, k=1, Lin=300,
                               epi=RES_SKIP, rs_split=H if rs else 0, y2_first=first, y2_mask=ymask, mask=True))
    # COUPLE: both signs, x1 from res (a flow's first touch of its input) and from y
    for sign in (1, -1):
        for res in ("none", "sep"):
            cs.append(case(f"couple-{sign}-{res}", Cin=48, Cout=96, k=1, Lin=300, epi=COUPLE, couple_sign=sign,
                           res=res, mask=True))
    # MAG: the spectrogram's framed rows, Lin = Lq + taps - 1, positive in_off0, frames where re = im = 0
    for Cout, k in ((34, 3), (162, 5)):
        cs.append(case(f"mag-{Cout}-k{k}", Cin=40, Cout=Cout, k=k, Lin=300 + k - 1, Lq=300, in_off0=0, epi=MAG,
                       bias=False, mask=True, zero_frames=True))
    cs.append(case("mag-offset", Cin=40, Cout=34, k=3, Lin=305, Lq=300, in_off0=2, epi=MAG, bias=False, mask=True,
                   zero_frames=True))
    # strided outputs: every phase, Lout not a multiple of the stride; the rows of the other phases keep the sentinel
    for s in (2, 3, 5):
        Lout = 96 * s + 1 + (s > 2)
        for ph in range(s):
            Lq = (Lout - ph + s - 1) // s
            cs.append(case(f"stride{s}-phase{ph}", Cin=9, Cout=17, k=3, Lin=Lq, Lq=Lq, out_stride=s, out_phase=ph,
                           Lout=Lout, pre_lrelu=1, in_off0=-1))
    return cs


SMEM_REFUSED = case("smem-200k-over", Cin=9, Cout=40, k=5, dil=1457, Lin=6000, Lq=300, in_off0=-2900)

# the decoder's upsamplers: the five stages of the full config and odd shapes (Cin, Cout, rate, k)
UPS_SHAPES = ((512, 256, 5, 11), (256, 128, 5, 11), (128, 64, 3, 7), (64, 32, 2, 4), (32, 16, 2, 4), (24, 12, 3, 3),
              (16, 8, 4, 8), (16, 8, 1, 3))
UPS_LINS = (1, 2, 257)
POST_CASES = [(C, k, L) for C in (16, 32) for k in (3, 7) for L in (511, 512, 513)]
COND_CASES = [(O, I, B) for I in (1, 31, 32, 33, 256) for O in (1, 512, 1536, 6144) for B in (1, 3)]


# ---- operands --------------------------------------------------------------------------------------------------------

def _grid(gen, n, shape, step):
    """Integers in [-n, n] times step."""
    return torch.randint(-n, n + 1, shape, generator=gen).to(torch.float32) * step


def lengths(B, L):
    return [L, max(1, L - 37), max(1, (2 * L) // 3)][:B] + [L] * max(0, B - 3)


def operands(c, layer):
    """fp32 CPU operands of a convolution case: x [B, Cin, Lin], w [Cout, Cin, k], bias [Cout] (reference order),
    bcond [B, Cout] (packed order), res [B, Cout, Lout], mask [B, Lout] (0 / 1), y_old [B, ych, Lout],
    y2_old [B, Cout - rs_split, Lout], slope."""
    g = torch.Generator().manual_seed(c["seed"] * 2 + (layer == "random"))
    B, Cin, Cout, k, Lin, Lout = c["B"], c["Cin"], c["Cout"], c["k"], c["Lin"], c["Lout"]
    ych, ny2 = ychannels(c), Cout - c["rs_split"] if c["epi"] == RES_SKIP else 0
    if layer == "exact":
        x = _grid(g, 128, (B, Cin, Lin), GRID_X)
        w = _grid(g, 4, (Cout, Cin, k), GRID_W)
        add = lambda shape, m: _grid(g, int(m / GRID_ADD), shape, GRID_ADD)
        slope = 0.0 if c["relu"] else EXACT_SLOPE
    else:
        x = torch.randn(B, Cin, Lin, generator=g)
        w = torch.randn(Cout, Cin, k, generator=g) / math.sqrt(Cin * k)
        add = lambda shape, m: torch.randn(shape, generator=g) * (m / 4)
        slope = 0.0 if c["relu"] else SLOPE
    if c["zero_frames"]:
        x[:, :, Lin // 3:Lin // 3 + k + 20] = 0
    mask = torch.zeros(B, Lout)
    for b, n in enumerate(lengths(B, Lout)):
        mask[b, :n] = 1
    return dict(x=x, w=w, bias=add((Cout,), BIAS_MAX) if c["bias"] else None,
                bcond=add((B, Cout), BCOND_MAX) if c["bcond"] else None,
                res=add((B, Cout, Lout), RES_MAX), mask=mask if c["mask"] else None,
                y_old=add((B, ych, Lout), OLD_MAX), y2_old=add((B, ny2, Lout), OLD_MAX), slope=slope)


def ups_operands(Cin, Cout, rate, k, B, Lin, layer, seed):
    """x [B, Cin, Lin] (>= 0 on exact operands: the load slope is 0.1), w [Cin, Cout, k], bias [Cout]."""
    g = torch.Generator().manual_seed(seed)
    if layer == "exact":
        return (_grid(g, 128, (B, Cin, Lin), GRID_X).abs(), _grid(g, 4, (Cin, Cout, k), GRID_W),
                _grid(g, int(BIAS_MAX / GRID_ADD), (Cout,), GRID_ADD))
    return (torch.randn(B, Cin, Lin, generator=g), torch.randn(Cin, Cout, k, generator=g) / math.sqrt(Cin * k / rate),
            0.1 * torch.randn(Cout, generator=g))


def post_operands(C, k, L, B, layer, seed):
    """x [B, C, L], w [C, k], slope."""
    g = torch.Generator().manual_seed(seed)
    if layer == "exact":
        return _grid(g, 128, (B, C, L), GRID_X), _grid(g, 4, (C, k), GRID_W), EXACT_SLOPE
    return torch.randn(B, C, L, generator=g), torch.randn(C, k, generator=g) / math.sqrt(C * k), SLOPE


def cond_operands(O, I, B, layer, seed):
    """W [O, I], bias [O], g [B, I]."""
    gen = torch.Generator().manual_seed(seed)
    if layer == "exact":
        return (_grid(gen, 4, (O, I), GRID_W), _grid(gen, int(BIAS_MAX / GRID_ADD), (O,), GRID_ADD),
                _grid(gen, 128, (B, I), GRID_X))
    return torch.randn(O, I, generator=gen) / math.sqrt(I), 0.1 * torch.randn(O, generator=gen), torch.randn(B, I, generator=gen)


# ---- references --------------------------------------------------------------------------------------------------------

def load(x, pre_lrelu, slope):
    """f(x) as the kernel stages it: leaky_relu in fp32 (v > 0 ? v : v * slope)."""
    x = x.to(torch.float32)
    if pre_lrelu:
        x = torch.where(x > 0, x, x * torch.tensor(slope, dtype=torch.float32))
    return x


def round_operand(t, fault):
    t = t.to(torch.float32).contiguous()
    if fault == "bf16":
        return t.to(torch.bfloat16).to(torch.float32)
    if fault == "tf32":     # 10 explicit mantissa bits, nearest (ties away, as cvt.rna.tf32.f32)
        b = t.view(torch.int32)
        return ((b + 0x1000) & ~0x1FFF).view(torch.float32)
    return t


def conv_acc(xf, w, Lq, in_off0, dil, fault=None):
    """acc [B, Cout, Lq] and S (sum of |products|) in float64: xf = f(x) [B, Cin, Lin], w [Cout, Cin, k]."""
    xf = round_operand(xf, fault).double()
    w = round_operand(w, fault).double()
    B, Cin, Lin = xf.shape
    k = w.shape[2]
    if fault == "tail_chunk" and Cin % CI_CHUNK:
        xf = xf.clone()
        xf[:, Cin - Cin % CI_CHUNK:] = 0
    if fault == "last_tap":
        w = w.clone()
        w[:, :, -1] = 0
    if fault == "in_off0":
        in_off0 += 1
    lo = in_off0
    hi = (Lq - 1) + in_off0 + (k - 1) * dil + 1        # input positions [lo, hi) are read
    left, right = max(0, -lo), max(0, hi - Lin)
    if fault == "right_clamp" and right:
        xp = torch.cat([F.pad(xf, (left, 0)), xf[:, :, -1:].expand(B, Cin, right)], 2)
    else:
        xp = F.pad(xf, (left, right))
    xp = xp[:, :, lo + left:hi + left]
    acc = F.conv1d(xp, w, dilation=dil)[:, :, :Lq]
    S = F.conv1d(xp.abs(), w.abs(), dilation=dil)[:, :, :Lq]
    return acc, S


def _tol(n, m, S):
    return gamma(n + m) * S


def conv_ref(c, op, layer, fault=None):
    """The launch's outputs in float64: {name: (value, tol, written (bool), S)}, each [B, ch, Lout], for y (and y2 for
    RES_SKIP).  tol is the gate of the layer at each written element: 0 where the exact layer knows the
    value exactly, the function-ulp bound for GATE / MAG on exact operands, the fp32 FMA bound on random operands."""
    B, Cout, Lq, Lout, epi = c["B"], c["Cout"], c["Lq"], c["Lout"], c["epi"]
    s, ph = c["out_stride"], c["out_phase"] + (1 if fault == "phase_off" else 0)
    exact = layer == "exact"
    n = c["Cin"] * c["k"]
    xf = load(op["x"], c["pre_lrelu"], op["slope"])
    acc, Sacc = conv_acc(xf, op["w"], Lq, c["in_off0"], c["dil"], fault)
    pos = torch.arange(Lq) * s + ph
    keep = pos < Lout
    pos = pos[keep]
    acc, Sacc = acc[:, :, keep], Sacc[:, :, keep]

    def at(t):   # [B, C, Lout] -> the rows this launch writes
        return t.double()[:, :, pos]

    mk = torch.ones(B, 1, pos.numel(), dtype=torch.float64)
    if op["mask"] is not None:
        m = op["mask"].double()
        if fault == "mask_bs_lout":   # row b read at b * Lout from the buffer laid out with rows of mask_bs
            flat = mask_buffer(c, op["mask"]).double()
            m = torch.stack([flat[b * Lout:(b + 1) * Lout] for b in range(B)])
        mk = m[:, pos].unsqueeze(1)
    # bias and bcond in the reference's channel order
    bias = op["bias"].double() if op["bias"] is not None else torch.zeros(Cout, dtype=torch.float64)
    if fault == "bias_twice":
        bias = 2 * bias
    bc = torch.zeros(B, Cout, dtype=torch.float64)
    if op["bcond"] is not None:
        bc = op["bcond"].double()
        if fault == "bcond_neighbour":
            bc = bc.roll(-1, 0)
        if c["gate_interleave"]:
            H = Cout // 2
            bc = torch.cat([bc[:, 0::2][:, :H], bc[:, 1::2][:, :H]], 1)
    v = acc + bias[None, :, None] + bc[:, :, None]
    Sv = Sacc + bias.abs()[None, :, None] + bc.abs()[:, :, None]
    out = {}

    def put(name, ch, val, tol, S, skip=0):
        V, T, SS = (torch.zeros(B, ch, Lout, dtype=torch.float64) for _ in range(3))
        Wr = torch.zeros(B, ch, Lout, dtype=torch.bool)
        V[:, :, pos], T[:, :, pos], SS[:, :, pos] = val, tol, S
        Wr[:, skip:, pos] = True
        out[name] = (V, T, Wr, SS)

    if epi == LINEAR:
        r = at(op["y_old"]) if c["res"] == "alias" else at(op["res"]) if c["res"] == "sep" else 0
        u = (v + r) * mk
        Su = (Sv + (r.abs() if c["res"] != "none" else 0)) * mk.abs()
        if c["acc_mode"] == ACC_SET:
            val, S = u, Su
        else:
            yo = at(op["y_old"])
            val, S = yo + u, yo.abs() + Su
            if c["acc_mode"] == ACC_ADD_DIV:
                nk = torch.tensor(float(c["nk"]), dtype=torch.float32)
                if exact:     # one IEEE division of an exact fp32 value
                    f32 = val.to(torch.float32)
                    val = (f32 * (1.0 / nk) if fault == "add_div_mul" else f32 / nk).double()
                else:
                    val = val / c["nk"]
                S = S / c["nk"]
        put("y", Cout, val, 0 * S if exact else _tol(n, 6, S), S)
    elif epi == GATE:
        H = Cout // 2
        if not c["gate_interleave"]:   # weights given in the packed order: output c = (v[2c], v[2c + 1])
            a, sg, Sa, Ss = v[:, 0::2], v[:, 1::2], Sv[:, 0::2], Sv[:, 1::2]
        else:
            a, sg, Sa, Ss = v[:, :H], v[:, H:], Sv[:, :H], Sv[:, H:]
        if fault == "gate_swap":
            a, sg = sg, a
        val = torch.tanh(a) * torch.sigmoid(sg)
        e = 0 if exact else _tol(n, 2, Sa) + _tol(n, 2, Ss) / 4
        put("y", H, val, e * (1 + 12 * U) + 12 * U * val.abs() + TINY, Sa + Ss / 4)
    elif epi == MAG:
        a, sg, Sa, Ss = acc[:, 0::2], acc[:, 1::2], Sacc[:, 0::2], Sacc[:, 1::2]
        eps = 0.0 if fault == "mag_no_eps" else MAG_EPS
        mag = torch.sqrt(a * a + sg * sg + eps)
        val = mag * mk
        ea, es = (0, 0) if exact else (_tol(n, 0, Sa), _tol(n, 0, Ss))
        tol = (ea + es + (ea * ea + es * es) / mag.clamp_min(TINY) + 4 * U * mag) * mk.abs()
        put("y", Cout // 2, val, tol + TINY, (Sa + Ss + mag) * mk.abs())   # (S: + the magnitude's own roundings)
    elif epi == RES_SKIP:
        rs = c["rs_split"]
        if rs:
            hs = at(op["y_old"])
            S = (hs.abs() + Sv[:, :rs]) * mk.abs()
            put("y", rs, (hs + v[:, :rs]) * mk, 0 * S if exact else _tol(n, 4, S), S)
        sk, Ssk = v[:, rs:], Sv[:, rs:]
        if not c["y2_first"] or fault == "y2_first_ignored":
            yo = at(op["y2_old"])
            sk, Ssk = yo + sk, yo.abs() + Ssk
        if c["y2_mask"] and fault != "skip_mask_missing":
            sk, Ssk = sk * mk, Ssk * mk.abs()
        # (rs_split 8 too large: the first 8 skip channels go to the state instead, and their skip rows stay unwritten)
        put("y2", Cout - rs, sk, 0 * Ssk if exact else _tol(n, 4, Ssk), Ssk, skip=8 if fault == "rs_split_8" else 0)
    elif epi == COUPLE:
        m = v * mk
        from_res = c["res"] == "sep" and fault != "x1_from_y"
        x1 = at(op["res"]) if from_res else at(op["y_old"])
        sign = -c["couple_sign"] if fault == "couple_sign" else c["couple_sign"]
        val = m + x1 * mk if sign > 0 else (x1 - m) * mk
        S = (Sv + x1.abs()) * mk.abs()
        put("y", Cout, val, 0 * S if exact else _tol(n, 6, S), S)
    return out


def mask_buffer(c, mask):
    """The mask as the GPU test lays it out: rows of mask_bs = Lout + 5, NaN beyond Lout."""
    B, Lout = mask.shape
    buf = torch.full((B, Lout + 5), float("nan"))
    buf[:, :Lout] = mask
    return buf.reshape(-1)


def phase_taps(k, rate):
    """The upsampler's polyphase split (csrc/run_tc.cu pack_upsampler): per phase r, (in_off0, [tap index j of the
    ConvTranspose1d weight for each of the n_r Conv1d taps])."""
    pad = (k - rate) // 2
    out = []
    for r in range(rate):
        j0 = (r + pad) % rate
        nr = (k - 1 - j0) // rate + 1
        cr = (r + pad - j0) // rate
        out.append((cr - nr + 1, [j0 + rate * (nr - 1 - jj) for jj in range(nr)]))
    return out


def upsample_ref(x, w, bias, rate, layer, fault=None):
    """y [B, Cout, Lin * rate] = conv_transpose1d(leaky_relu(x, 0.1)) + bias as the polyphase launches compute it, and
    the gate (0 on exact operands) and S.  w [Cin, Cout, k]."""
    B, Cin, Lin = x.shape
    Cout, k = w.shape[1], w.shape[2]
    xf = load(x, 1, SLOPE)
    y = torch.zeros(B, Cout, Lin * rate, dtype=torch.float64)
    tol, SS = torch.zeros_like(y), torch.zeros_like(y)
    for r, (off, taps) in enumerate(phase_taps(k, rate)):
        if fault == "ups_taps_reversed" and r == 0:
            taps = taps[::-1]
        wc = w[:, :, taps].permute(1, 0, 2)                       # as a Conv1d weight [Cout][Cin][n_r]
        Lq = (Lin * rate - r + rate - 1) // rate
        acc, S = conv_acc(xf, wc, Lq, off, 1, fault if fault in ("bf16", "tf32") else None)
        y[:, :, r::rate] = acc + bias.double()[None, :, None]
        SS[:, :, r::rate] = S + bias.double().abs()[None, :, None]
        if layer != "exact":
            tol[:, :, r::rate] = _tol(Cin * len(taps), 1, SS[:, :, r::rate])
    return y, tol, SS


def post_ref(x, w, slope, n0, n1, layer, fault=None):
    """wav [B, n1 - n0] = tanh(conv1d(leaky_relu(x, slope), w, padding (k - 1) / 2)) at samples [n0, n1), the gate and S."""
    B, C, L = x.shape
    k = w.shape[-1]
    xf = load(x, 1, slope)
    s, S = conv_acc(xf, w.reshape(1, C, k), L, -((k - 1) // 2), 1, fault if fault in ("bf16", "tf32") else None)
    lo = 0 if fault == "post_ignores_n0" else n0
    s, S = s[:, 0, lo:lo + n1 - n0], S[:, 0, lo:lo + n1 - n0]
    val = torch.tanh(s)
    e = 0 if layer == "exact" else _tol(C * k, 0, S)
    return val, e * (1 + 4 * U) + 4 * U * val.abs() + TINY, S


def cond_ref(W, bias, g, layer):
    """out [B, O] = bias + g @ W^T, the gate and S (lane chains of ceil(I / 32) FMAs, a five-level shuffle tree, the bias)."""
    W, g = W.double(), g.double()
    b = bias.double() if bias is not None else torch.zeros(W.shape[0], dtype=torch.float64)
    val = g @ W.T + b
    S = g.abs() @ W.abs().T + b.abs()
    n = -(-W.shape[1] // 32) + 5 + 1
    return val, (0 * S if layer == "exact" else _tol(n, 0, S)), S


def rejects(got, want, tol):
    """A comparator's verdict, and the worst |got - want| / tol over the elements (inf where tol = 0 and they differ)."""
    d = (got.double() - want.double()).abs()
    d = torch.where(torch.isnan(d), torch.full_like(d, float("inf")), d)
    r = d / tol.clamp_min(TINY) if tol is not None else d
    bad = (d > tol) if tol is not None else (d > 0)
    return bool(bad.any()), float(r.max()) if r.numel() else 0.0


def expected(init, val, written):
    """The buffer region [B, ch, Lout] a launch leaves: val where it writes, the initial content elsewhere."""
    return torch.where(written, val, init.double())


def compare(got, init, val, tol, written):
    """(ok, worst |got - val| / tol on the written elements): written elements within tol (tol = 0: equal, +-0 alike),
    every other element bit-identical to its initial content."""
    got = got.double()
    d = (got - val).abs()
    d = torch.where(torch.isnan(d), torch.full_like(d, float("inf")), d)
    ok_w = bool((d[written] <= tol[written]).all())
    un = ~written
    g32, i32 = got.to(torch.float32)[un].contiguous(), init.to(torch.float32)[un].contiguous()
    ok_u = torch.equal(g32.view(torch.int32), i32.view(torch.int32))
    ratio = float((d[written] / tol[written].clamp_min(TINY)).max()) if written.any() else 0.0
    return ok_w and ok_u, ratio
