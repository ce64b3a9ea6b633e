"""The fused ResBlock1 kernels (csrc/pair_tc.cuh, rb_tc.cuh, rp_tc.cuh) on exact operands (tests/resblock_reference.py):
the first convolution of the live pair is exact, so the intermediate's bf16 rounding and each kernel's leaky_relu are
known bit for bit and out_f32 is gated at a few fp32 ulp of S at every element; raw and act are checked bit for bit
against the kernel's own formulas from out_f32.  The whole-resblock kernels are tested one pair slot at a time.

Every output is a caller buffer pre-filled with NaN and followed by guard elements: every valid element must be written
and nothing past the end.  The floors (worst rel_err over this file, relative to S) and the gates are in
resblock_reference.EPS; the module prints the floors it measures."""
import ctypes

import pytest
import torch

import resblock_reference as R
from conv_reference import bits_equal, rel_err

pytestmark = pytest.mark.gpu

GUARD = 1000
DILS = (1, 3, 5)
FLOORS = {}


@pytest.fixture(scope="module", autouse=True)
def _print_floors():
    yield
    for kind in sorted(FLOORS):
        print(f"measured floor {kind} ({2 if kind == 'rp_x3' else 1} plane{'s' if kind == 'rp_x3' else ''}): "
              f"{FLOORS[kind]:.2e} x S (gate {R.EPS[kind]:.1e})")


def _lib():
    from visinger_b200 import _lib
    return _lib


def _buffer(n, dtype, dev):
    return torch.full((n + GUARD,), float("nan"), dtype=dtype, device=dev)


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _written(buf, n, what):
    """Elements [0, n) all written (no NaN left), the guard past them untouched."""
    buf = buf.cpu()
    assert not bool(torch.isnan(buf[:n].float()).any()), f"{what}: elements left unwritten"
    assert bits_equal(buf[n:], torch.full((GUARD,), float("nan"), dtype=buf.dtype)), f"{what}: written past the end"
    return buf[:n]


def _verify(kind, f32, raw, act, shape, want, S, label):
    """Gate out_f32 against the reference, raw / act bit for bit against the kernel's formulas; returns the outputs."""
    B, L, C = shape
    npl = 2 if kind == "rp_x3" else 1
    n = B * L * C
    out = _written(f32, n, f"{label} out_f32").view(B, L, C)
    e = rel_err(out, want, S)
    FLOORS[kind] = max(FLOORS.get(kind, 0.0), e)
    print(f"{label}: rel {e:.2e} x S (gate {R.EPS[kind]:.1e})")
    assert e <= R.EPS[kind], f"{label}: out_f32 off the float64 reference by {e:.3e} x S"
    got = []
    for buf, form, what in ((raw, R.out_raw, "raw"), (act, R.out_act, "act")):
        if buf is None:
            got.append(None)
            continue
        w = form(kind, out)
        g = _written(buf, npl * n, f"{label} {what}").view(w.shape)
        assert bits_equal(g, w), f"{label}: out_{what} differs from the kernel's formula at {int((g != w).sum())} elements"
        got.append(g)
    return out, got[0], got[1]


# ---- the fused pair (pair_tc.cuh) ------------------------------------------------------------------------------------

# the decoder's launches of the pair (run_tc.cu generator_forward_tc): a non-final pair writes the activated stream; the
# last pair of the first chain starts the running sum (raw), of a middle chain adds to it, of the last chain adds it, scales
# and writes the stage output
PAIR_FORMS = {"inner": (False, 1.0, ("act",), "RES_ACT"), "sum0": (False, 1.0, ("raw",), "LINEAR"),
              "sum": (True, 1.0, ("raw",), "LINEAR"), "final": (True, 1.0 / 3.0, ("act",), "LINEAR")}


def _pair_plan(C, k, dil, L, n_adds=2, n_outs=1):
    """vsg_debug_pair_plan: (blocks per tile, valid rows per tile, tiles per utterance) of the pair kernel."""
    L_ = _lib().lib()
    L_.vsg_debug_pair_plan.argtypes = [ctypes.c_int32] * 6 + [ctypes.POINTER(ctypes.c_int32)]
    L_.vsg_debug_pair_plan.restype = ctypes.c_int
    out = (ctypes.c_int32 * 3)()
    assert L_.vsg_debug_pair_plan(C, k, dil, L, n_adds, n_outs, out) == 0, (C, k, dil, L)
    return tuple(out)


def _pair_V(C, k, dil):
    return _pair_plan(C, k, dil, 4096)[1]


def _run_pair(xa, conv, dev, add0, add0_is_act, add1, scale, outs, f32):
    w1, b1, w2, b2, dil = conv
    B, L, C = xa.shape
    n = B * L * C
    bufs = {o: _buffer(n, torch.bfloat16, dev) for o in outs}
    out_f32 = _buffer(n, torch.float32, dev) if f32 else None
    img = _lib().debug_pair_tc(xa.to(dev), w1, b1, w2, b2, dil, add0=add0.to(dev) if add0 is not None else None,
                               add0_is_act=int(add0_is_act), add1=add1.to(dev) if add1 is not None else None, scale=scale,
                               out_raw=bufs.get("raw"), out_act=bufs.get("act"), out_f32=out_f32)
    return img, out_f32, bufs.get("raw"), bufs.get("act")


def _pair_case(C, k, dil, L, add0_kind, dev):
    g = torch.Generator().manual_seed(C * 1000 + k * 100 + dil * 10 + L)
    B = 3
    xa = R.exact_input(B, L, C, g)
    w1, b1 = R.exact_conv1(C, k, g)
    w2, b2 = R.dense_conv2(C, k, g)
    add1 = R.running_sum(B, L, C, g)
    add0 = xa if add0_kind == "act" else R.running_sum(B, L, C, g)
    conv = (w1, b1, w2, b2, dil)
    sig = _lib().EPI_SIG
    for form, (use_add1, scale, outs, image) in PAIR_FORMS.items():
        a1 = add1 if use_add1 else None
        want, S = R.reference("pair", xa, *conv, add0=add0, add0_is_act=add0_kind == "act", add1=a1, scale=scale)
        label = f"pair C={C} k={k} d={dil} L={L} add0={add0_kind} {form}"
        # (the form's own output: with two adds the pair has room for one output tile at C = 32, k >= 7)
        img, f32, raw, act = _run_pair(xa, conv, dev, add0, add0_kind == "act", a1, scale, outs, True)
        assert img == sig["GENERIC"], label
        _, graw, gact = _verify("pair", f32, raw, act, (B, L, C), want, S, label)
        # the image the decoder launches, without the fp32 copy: the same bits as the generic one
        img, _, raw, act = _run_pair(xa, conv, dev, add0, add0_kind == "act", a1, scale, outs, False)
        assert img == sig[image if add0_kind == "act" else "LINEAR"], (label, img)
        for buf, ref, what in ((raw, graw, "raw"), (act, gact, "act")):
            if buf is not None:
                assert bits_equal(_written(buf, B * L * C, f"{label} {what}").view(B, L, C), ref), f"{label}: {what} image"
    # two calls, same bits
    _, f1, _, _ = _run_pair(xa, conv, dev, add0, add0_kind == "act", None, 1.0, ("act",), True)
    _, f2, _, _ = _run_pair(xa, conv, dev, add0, add0_kind == "act", None, 1.0, ("act",), True)
    assert bits_equal(f1.cpu(), f2.cpu())


PAIR_CASES = [(C, k, d) for C in (16, 32) for k in (3, 7, 11) for d in DILS]


@pytest.mark.parametrize("add0_kind", ["act", "raw"])
@pytest.mark.parametrize("C,k,dil", PAIR_CASES)
def test_pair_exact(cuda_device, C, k, dil, add0_kind):
    """The fused pair at every (C, k, dilation) of the model's C = 16 / 32 stages, with the residual taken from the
    activated stream (the decoder's form) and as a raw add, in the three epilogue forms the decoder launches, B = 3 and
    a ragged last tile."""
    V = _pair_V(C, k, dil)
    _pair_case(C, k, dil, 2 * V + 37 + 8 * k + dil, add0_kind, cuda_device)


@pytest.mark.parametrize("C", [16, 32])
@pytest.mark.parametrize("where", ["tiles", "tiles+1", "tiles-1", "shortest"])
def test_pair_tile_edges(cuda_device, C, where):
    """Lengths at the tile geometry vsg_debug_pair_plan reports: exactly three tiles, one row more or less, and the
    shortest length the kernel takes (128 mb rows, two tiles)."""
    k, dil = 7, 3
    mb, V, _ = _pair_plan(C, k, dil, 4096)
    L = {"tiles": 3 * V, "tiles+1": 3 * V + 1, "tiles-1": 3 * V - 1, "shortest": 128 * mb}[where]
    assert _pair_plan(C, k, dil, L)[2] == {"tiles": 3, "tiles+1": 4, "tiles-1": 3, "shortest": 2}[where]
    _pair_case(C, k, dil, L, "act", cuda_device)


# ---- the whole-resblock kernels (rb_tc.cuh, rp_tc.cuh) ----------------------------------------------------------------

def _run_resblock(xa, ws, bs, dils, add1, scale, max_mb, sets, dev):
    x3 = bool(sets & 2048)
    B, L, C = xa.shape[-3:]
    n = B * L * C
    npl = 2 if x3 else 1
    f32 = _buffer(n, torch.float32, dev)
    raw = _buffer(npl * n, torch.bfloat16, dev)
    act = _buffer(npl * n, torch.bfloat16, dev)
    wh = torch.stack([w.float() for w in ws]).contiguous()
    bh = torch.stack([b.float() for b in bs]).contiguous()
    dl = (ctypes.c_int32 * len(dils))(*dils)
    xd = xa.to(dev).contiguous()
    a1 = add1.to(dev).contiguous() if add1 is not None else None
    torch.cuda.synchronize(dev)
    rc = _lib().lib().vsg_debug_resblock_bf16(xd.data_ptr(), wh.data_ptr(), bh.data_ptr(), len(dils), dl, _ptr(a1),
                                              float(scale), f32.data_ptr(), raw.data_ptr(), act.data_ptr(), B, L, C,
                                              ws[0].shape[2], int(max_mb), int(sets), dev.index or 0)
    _lib().check(rc, "vsg_debug_resblock_bf16")
    return f32, raw, act


def _slot_case(kind, sets, C, k, dils, q, B, L, max_mb, dev, nonneg=None):
    """Slot q of a resblock: the live pair against the reference, with and without the running sum and scale; the same
    run with the trailing zero pairs cut off gives the same bits; two calls give the same bits."""
    g = torch.Generator().manual_seed(C * 7919 + k * 131 + q * 17 + L + sets)
    x3 = kind == "rp_x3"
    xa = R.exact_input(B, L, C, g, nonneg=q > 0 if nonneg is None else nonneg, x3=x3)
    if q > 0:
        assert R.slot_input_check(kind, xa)
    ws, bs = R.slot_weights(C, k, len(dils), q, g)
    add1 = R.running_sum(B, L, C, g, x3=x3)
    conv = (ws[2 * q], bs[2 * q], ws[2 * q + 1], bs[2 * q + 1], dils[q])
    tag = f"{kind}[{sets}] C={C} k={k} dils={dils} q={q} B={B} L={L} max_mb={max_mb}"
    outs = {}
    for a1, scale in ((add1, 1.0 / 3.0), (None, 1.0)):
        want, S = R.reference(kind, xa, *conv, add1=a1, scale=scale)
        f32, raw, act = _run_resblock(xa, ws, bs, dils, a1, scale, max_mb, sets, dev)
        outs[a1 is None] = _verify(kind, f32, raw, act, (B, L, C), want, S, f"{tag} add1={a1 is not None}")
    if q + 1 < len(dils):
        cut = _run_resblock(xa, ws[:2 * q + 2], bs[:2 * q + 2], dils[:q + 1], None, 1.0, max_mb, sets, dev)
        for got, ref in zip(cut, outs[True]):
            assert bits_equal(got.cpu()[:ref.numel()].view(ref.shape), ref), f"{tag}: trailing zero pairs changed the bits"
    again = _run_resblock(xa, ws, bs, dils, None, 1.0, max_mb, sets, dev)
    for got, ref in zip(again, outs[True]):
        assert bits_equal(got.cpu()[:ref.numel()].view(ref.shape), ref), f"{tag}: a second call gave other bits"


def _rp_plan(C, k, dils, L, variant):
    """vsg_debug_rp_plan: (blocks per tile, halo, valid steps per tile); variant 0 plain, 1 split-bf16, 2 two CTAs."""
    L_ = _lib().lib()
    L_.vsg_debug_rp_plan.argtypes = [ctypes.c_int32] * 3 + [ctypes.POINTER(ctypes.c_int32), ctypes.c_int32, ctypes.c_int32,
                                                             ctypes.POINTER(ctypes.c_int32)]
    L_.vsg_debug_rp_plan.restype = ctypes.c_int
    out = (ctypes.c_int32 * 8)()
    assert L_.vsg_debug_rp_plan(C, k, len(dils), (ctypes.c_int32 * len(dils))(*dils), L, variant, out) == 0
    return out[0], out[1], out[2]


def _plan_variant(sets):
    return 1 if sets & 2048 else 2 if sets & 4096 else 0


def _ragged(C, k, dils, sets):
    """Two tiles and a part of a third at the kernel's own tile size, a whole number of row-packed rows."""
    S = 64 // C
    _, _, V = _rp_plan(C, k, dils, 1 << 16, _plan_variant(sets))
    return 2 * V + (V // 3) // S * S


RB_CASES = [(C, k, q) for C in (16, 32, 64) for k in (3, 7, 11) for q in range(3)]


@pytest.mark.parametrize("C,k,q", RB_CASES)
def test_rb_slot_exact(cuda_device, C, k, q):
    """rb_tc (default epilogue sets) at every (C, k) of the model's C <= 64 stages, each pair slot of a three-pair block
    with its own dilation; tiles capped at 2 / 4 blocks or as many as fit."""
    _slot_case("rb", 0, C, k, DILS, q, 3, 700 + 111 * q + 13 * k, (0, 2, 4)[(q + k) % 3], cuda_device)


RP_VARIANTS = [256, 256 | 512, 256 | 1024, 256 | 4096]
RP_CASES = [(C, k, q) for C in (16, 32) for k in (3, 7, 11) for q in range(3)]
RP_MAX_MB = {(C, k, q): 1 + (q + k // 4 + C // 16) % 4 for C, k, q in RP_CASES}
assert set(RP_MAX_MB.values()) == {1, 2, 3, 4} and all(len({RP_MAX_MB[(C, k, q)] for q in range(3)}) == 3
                                                         for C, k, _ in RP_CASES)


@pytest.mark.parametrize("C,k,q", RP_CASES)
@pytest.mark.parametrize("sets", RP_VARIANTS)
def test_rp_slot_exact(cuda_device, sets, C, k, q):
    """rp_tc in its block-Toeplitz form (256), tap by tap (| 512), two epilogue sets per block (| 1024) and two CTAs per
    SM (| 4096), every (C, k) of the C = 16 / 32 stages and every pair slot, ragged last tiles, tiles capped at 1 .. 4
    blocks (the two-CTA form takes at most 2)."""
    _slot_case("rp", sets, C, k, DILS, q, 3, _ragged(C, k, DILS, sets), RP_MAX_MB[(C, k, q)], cuda_device)


# the odd shapes of test_gpu_round2.RP_CASES: a kernel size the model does not use, two pairs, one pair, dilations 2, 1
RP_ODD = [(16, 5, (1, 2)), (16, 3, (1,)), (32, 9, (2, 1))]


@pytest.mark.parametrize("C,k,dils", RP_ODD)
@pytest.mark.parametrize("sets", RP_VARIANTS)
def test_rp_odd_shapes_exact(cuda_device, sets, C, k, dils):
    for q in range(len(dils)):
        _slot_case("rp", sets, C, k, dils, q, 3, _ragged(C, k, dils, sets), 0, cuda_device)


@pytest.mark.parametrize("k,q", [(k, q) for k in (3, 7, 11) for q in range(3)])
def test_rp_c64_direct_exact(cuda_device, k, q):
    """rp_tc at C = 64: one time step per row, every convolution in the direct (tap by tap) form."""
    _slot_case("rp", 256, 64, k, DILS, q, 3, 900 + 37 * k + q, 0, cuda_device)


@pytest.mark.parametrize("C,k,q", RP_CASES)
@pytest.mark.parametrize("sets", [256 | 2048, 256 | 512 | 2048])
def test_rp_x3_slot_exact(cuda_device, sets, C, k, q):
    """rp_tc's split-bf16 instantiation (the bf16x3 decoder): planar two-plane input, running sum and raw output, rows
    [hi | lo] of the activated output; block-Toeplitz form and tap by tap, 1 or 2 blocks per tile."""
    _slot_case("rp_x3", sets, C, k, DILS, q, 3, _ragged(C, k, DILS, sets), 1 + (q + k) % 2, cuda_device)


GEOMETRY = ["tiles", "tiles+row", "tiles-row", "ragged", "below_halo"]


@pytest.mark.parametrize("where", GEOMETRY)
@pytest.mark.parametrize("C", [16, 32])
@pytest.mark.parametrize("sets", [256, 256 | 4096, 256 | 2048])
def test_rp_tile_edges(cuda_device, sets, C, where):
    """Lengths at the tile geometry vsg_debug_rp_plan reports: exactly two tiles, one row-packed row (64 / C steps) more
    or less, a ragged last tile, and an utterance shorter than the halo; slot 0 with a signed input (the residual's
    negative branch), k = 7."""
    k = 7
    S = 64 // C
    _, H, V = _rp_plan(C, k, DILS, 1 << 16, _plan_variant(sets))
    L = {"tiles": 2 * V, "tiles+row": 2 * V + S, "tiles-row": 2 * V - S, "ragged": V + V // 2 // S * S,
         "below_halo": (H - 1) // S * S}[where]
    kind = "rp_x3" if sets & 2048 else "rp"
    _slot_case(kind, sets, C, k, DILS, 0, 3, L, 0, cuda_device)
    if where == "tiles":
        _slot_case(kind, sets, C, k, DILS, 2, 3, L, 0, cuda_device)


@pytest.mark.parametrize("C,k", [(C, k) for C in (16, 32) for k in (3, 7, 11)])
@pytest.mark.parametrize("sets", [256, 256 | 512, 256 | 1024])
def test_rp_three_block_tiles(cuda_device, sets, C, k):
    """Utterances between two and three tiles' worth of valid steps, where the default plan (no cap) runs 3-block tiles:
    the planner picks mb = 3 there, and slots 0 and 2 are exact."""
    S = 64 // C
    mb4, H, V4 = _rp_plan(C, k, DILS, 1 << 16, 0)
    assert mb4 == 4
    V2, V3 = V4 - 256 * S, V4 - 128 * S
    L = (V2 + V3) // 2 // S * S
    assert _rp_plan(C, k, DILS, L, 0)[0] == 3, (C, k, L)
    for q in (0, 2):
        _slot_case("rp", sets, C, k, DILS, q, 3, L, 0, cuda_device)
