"""CPU: the float64 statements of the fp32 FFMA kernels (tests/conv_f32_reference.py) against torch, the exact-operand
bound over the GPU case matrix, the rejection of every named fault by the gate of the layer that targets it, the tile plan
of vsg_debug_conv_f32_plan, and the argument errors of the fp32 hooks (none of which needs a device).

On the exact layer every structural fault changes at least one element beyond the gate (0 for the exactly known
epilogues), ADD_DIV as a multiply by fp32(1/3) included.  On the random layer the worst |fault - reference| / gate is
527 for TF32 operands, 4.6e3 for bf16 operands and 6e4 or more for every structural fault (the test prints each)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import conv_f32_reference as R

C = R.case


# ---- the references against torch --------------------------------------------------------------------------------------

@pytest.mark.parametrize("k,dil,Cin,Cout,pre", [(1, 1, 5, 7, 0), (3, 1, 9, 16, 1), (5, 3, 8, 33, 1), (7, 1, 3, 2, 0)])
def test_conv_reference_matches_conv1d(k, dil, Cin, Cout, pre):
    c = C(f"ref-{k}-{dil}", Cin=Cin, Cout=Cout, k=k, dil=dil, Lin=50, pre_lrelu=pre)
    op = R.operands(c, "random")
    V, _, Wr, _ = R.conv_ref(c, op, "random")["y"]
    xf = F.leaky_relu(op["x"].double(), R.SLOPE) if pre else op["x"].double()
    want = F.conv1d(xf, op["w"].double(), op["bias"].double(), padding=(k - 1) * dil // 2, dilation=dil)
    assert bool(Wr.all())
    assert torch.allclose(V, want, rtol=0, atol=1e-6)      # f in fp32 (v * 0.1f) against float64 leaky_relu
    op["x"] = op["x"].abs()                                 # no negative loads: the same to float64 rounding
    V, _, _, _ = R.conv_ref(c, op, "random")["y"]
    want = F.conv1d(op["x"].double(), op["w"].double(), op["bias"].double(), padding=(k - 1) * dil // 2, dilation=dil)
    assert torch.allclose(V, want, rtol=0, atol=1e-12)


def test_strided_reference_places_rows_at_their_phase():
    c = C("ref-stride", Cin=4, Cout=3, k=3, Lin=20, Lq=20, out_stride=3, out_phase=2, Lout=61, in_off0=-1)
    op = R.operands(c, "random")
    V, _, Wr, _ = R.conv_ref(c, op, "random")["y"]
    dense = F.conv1d(op["x"].double(), op["w"].double(), op["bias"].double(), padding=1)
    assert torch.allclose(V[:, :, 2::3], dense, atol=1e-12) and bool(Wr[:, :, 2::3].all())
    assert not bool(Wr[:, :, 0::3].any()) and not bool(Wr[:, :, 1::3].any())


@pytest.mark.parametrize("Cin,Cout,rate,k", [(8, 4, 5, 11), (6, 3, 3, 7), (4, 2, 2, 4), (3, 5, 4, 8), (2, 2, 1, 3)])
def test_upsample_reference_matches_conv_transpose1d(Cin, Cout, rate, k):
    for Lin in (1, 2, 13):
        x, w, b = R.ups_operands(Cin, Cout, rate, k, 2, Lin, "random", 3)
        y, _, _ = R.upsample_ref(x, w, b, rate, "random")
        want = F.conv_transpose1d(F.leaky_relu(R.load(x, 1, R.SLOPE).double(), 1.0), w.double(), b.double(), stride=rate,
                                  padding=(k - rate) // 2)
        assert y.shape == want.shape and torch.allclose(y, want, rtol=0, atol=1e-12)


def test_post_and_cond_references_match_torch():
    x, w, slope = R.post_operands(16, 7, 300, 2, "random", 4)
    v, _, _ = R.post_ref(x, w, slope, 40, 290, "random")
    want = torch.tanh(F.conv1d(R.load(x, 1, slope).double(), w.double().reshape(1, 16, 7), padding=3))[:, 0, 40:290]
    assert torch.allclose(v, want, rtol=0, atol=1e-12)
    W, b, g = R.cond_operands(33, 40, 3, "random", 5)
    v, _, _ = R.cond_ref(W, b, g, "random")
    assert torch.allclose(v, F.linear(g.double(), W.double(), b.double()), rtol=0, atol=1e-12)


def test_tf32_rounding_keeps_ten_mantissa_bits():
    t = torch.tensor([1 + 2 ** -10, 1 + 2 ** -11, 1 + 2 ** -11 + 2 ** -20, 1 + 2 ** -12])
    assert R.round_operand(t, "tf32").tolist() == [1 + 2 ** -10, 1 + 2 ** -10, 1 + 2 ** -10, 1.0]


# ---- the exact-operand bound ---------------------------------------------------------------------------------------------

def test_exact_bound_holds_for_every_gpu_case():
    """Every partial sum of every GPU case stays below 2^24 units of the 2^-15 grid, so the exact layer is exact."""
    lim = 2.0 ** 24
    for c in R.gpu_cases() + [R.SMEM_REFUSED]:
        assert R.conv_exact_bound(c) < lim, c["name"]
    for Cin, Cout, rate, k in R.UPS_SHAPES:
        assert R.exact_bound(Cin * -(-k // rate), R.BIAS_MAX) < lim
    for Cc, k, L in R.POST_CASES:
        assert R.exact_bound(Cc * k, 0) < lim
    for O, I, B in R.COND_CASES:
        assert R.exact_bound(I, R.BIAS_MAX) < lim
    # and the largest shipped contraction (Cin * k = 256 * 11) is in the matrix while Cin = 513 at k = 11 is not
    assert any(c["Cin"] * c["k"] == 256 * 11 for c in R.gpu_cases())
    assert R.exact_bound(513 * 11, 8) >= lim


def test_exact_operands_sit_on_their_grids():
    c = C("grid", Cin=9, Cout=16, k=3, Lin=40, bcond=True, res="sep")
    op = R.operands(c, "exact")
    for name, step in (("x", R.GRID_X), ("w", R.GRID_W), ("bias", R.GRID_ADD), ("bcond", R.GRID_ADD),
                       ("res", R.GRID_ADD), ("y_old", R.GRID_ADD)):
        t = op[name].double() / step
        assert torch.equal(t, t.round()), name
    assert op["x"].abs().max() <= R.X_MAX and op["w"].abs().max() <= R.W_MAX


# ---- named faults ----------------------------------------------------------------------------------------------------------

_LIN = dict(Cin=9, Cout=16, k=3, Lin=80, pre_lrelu=1)
FAULT_CASES = {
    "tail_chunk": C("f-tail", **_LIN),
    "last_tap": C("f-tap", **_LIN),
    "in_off0": C("f-off", **_LIN),
    "right_clamp": C("f-clamp", **_LIN),
    "mask_bs_lout": C("f-mask", **_LIN, mask=True),
    "bcond_neighbour": C("f-bcond", **_LIN, bcond=True),
    "gate_swap": C("f-gate", Cin=8, Cout=32, k=5, Lin=80, epi=R.GATE, bcond=True, gate_interleave=1),
    "bias_twice": C("f-bias", **_LIN),
    "y2_first_ignored": C("f-first", Cin=16, Cout=32, k=1, Lin=80, epi=R.RES_SKIP, rs_split=16, y2_first=1, mask=True),
    "skip_mask_missing": C("f-skipmask", Cin=16, Cout=16, k=1, Lin=80, epi=R.RES_SKIP, rs_split=0, y2_mask=1, mask=True),
    "rs_split_8": C("f-split", Cin=16, Cout=32, k=1, Lin=80, epi=R.RES_SKIP, rs_split=16, mask=True),
    "couple_sign": C("f-sign", Cin=16, Cout=16, k=1, Lin=80, epi=R.COUPLE, couple_sign=-1, res="sep", mask=True),
    "x1_from_y": C("f-x1", Cin=16, Cout=16, k=1, Lin=80, epi=R.COUPLE, couple_sign=1, res="sep", mask=True),
    "add_div_mul": C("f-div", Cin=16, Cout=16, k=3, Lin=200, acc_mode=R.ACC_ADD_DIV, nk=3, res="sep", pre_lrelu=1),
    "mag_no_eps": C("f-mag", Cin=12, Cout=10, k=3, Lin=82, Lq=80, in_off0=0, epi=R.MAG, bias=False, mask=True,
                    zero_frames=True),
    "phase_off": C("f-phase", Cin=9, Cout=17, k=3, Lin=33, Lq=33, out_stride=3, out_phase=1, Lout=100, in_off0=-1),
    "bf16": C("f-bf16", Cin=8, Cout=16, k=1, Lin=80),
    "tf32": C("f-tf32", Cin=8, Cout=16, k=1, Lin=80),
}


def _rejection(fault, layer):
    """(rejected, margin) of a fault under the layer's gate: margin = worst |fault - reference| / gate."""
    if fault == "ups_taps_reversed":
        x, w, b = R.ups_operands(16, 8, 4, 8, 2, 9, layer, 6)
        y, tol, _ = R.upsample_ref(x, w, b, 4, layer)
        yf, _, _ = R.upsample_ref(x, w, b, 4, layer, fault)
        return R.rejects(yf, y, tol)
    if fault == "post_ignores_n0":
        x, w, slope = R.post_operands(16, 7, 300, 2, layer, 7)
        v, tol, _ = R.post_ref(x, w, slope, 100, 260, layer)
        vf, _, _ = R.post_ref(x, w, slope, 100, 260, layer, fault)
        return R.rejects(vf, v, tol)
    c = FAULT_CASES[fault]
    op = R.operands(c, layer)
    clean, bad = R.conv_ref(c, op, layer), R.conv_ref(c, op, layer, fault)
    verdict, margin = False, 0.0
    for name, (V, T, Wr, _) in clean.items():
        init = torch.full_like(V, 12345.0)
        want = R.expected(init, V, Wr)
        got = R.expected(init, bad[name][0], bad[name][2])
        d = (got - want).abs()
        d = torch.where(torch.isnan(d), torch.full_like(d, float("inf")), d)
        verdict |= bool((d > T).any())
        margin = max(margin, float((d / T.clamp_min(R.TINY)).max()))
    return verdict, margin


@pytest.mark.parametrize("fault", sorted(R.FAULTS))
def test_named_fault_is_rejected(fault):
    for layer in R.FAULTS[fault]:
        rejected, margin = _rejection(fault, layer)
        print(f"fault {fault:18s} {layer:6s} " + (f"margin {margin:.3g}" if layer == "random" else "differs"))
        assert rejected, (fault, layer)
        if layer == "random":
            assert margin >= 4, (fault, margin)


# ---- the tile plan and the argument errors -------------------------------------------------------------------------------

def _lib():
    from visinger_b200 import _lib
    return _lib


def test_conv_f32_plan_configurations_and_shared_memory():
    L = _lib()
    assert L.debug_conv_f32_plan(16, 5, 1)[:2] == (2, 4) and L.debug_conv_f32_plan(17, 5, 1)[:2] == (4, 2)
    assert L.debug_conv_f32_plan(32, 5, 1)[:2] == (4, 2) and L.debug_conv_f32_plan(33, 5, 1)[:2] == (8, 1)
    assert L.debug_conv_f32_plan(1, 1, 1) == (2, 4, 4 * 8 * (1024 + 16))
    # Cout > 32, k = 2: 4 * 8 * ((256 + dil) + 2 * 64) bytes, 48 KB at dil = 1152
    assert L.debug_conv_f32_plan(40, 2, 1152) == (8, 1, 48 * 1024)
    assert L.debug_conv_f32_plan(40, 2, 1153) == (8, 1, 48 * 1024 + 32)
    # k = 5: 4 * 8 * ((256 + 4 dil) + 5 * 64), 200 KB at dil = 1456; one more is refused
    assert L.debug_conv_f32_plan(40, 5, 1456) == (8, 1, 200 * 1024)
    assert L.debug_conv_f32_plan(40, 5, 1457) is None
    assert L.lib().vsg_debug_conv_f32_plan(40, 5, 1457, (ctypes.c_int32 * 3)()) == -4
    assert L.lib().vsg_debug_conv_f32_plan(0, 5, 1, (ctypes.c_int32 * 3)()) == -1
    assert L.lib().vsg_debug_conv_f32_plan(16, 5, 1, None) == -1
    for c in R.gpu_cases():
        assert L.debug_conv_f32_plan(c["Cout"], c["k"], c["dil"]) is not None, c["name"]
    c = R.SMEM_REFUSED
    assert L.debug_conv_f32_plan(c["Cout"], c["k"], c["dil"]) is None


def _desc(**kw):
    L = _lib()
    d = dict(x=1, w=1, y=1, x_bs=64, y_bs=64, x_cs=64, y_cs=64, B=1, Cin=1, Lin=64, Cout=1, k=1, dil=1, Lq=64,
             out_stride=1, Lout=64, couple_sign=1, acc_div=1.0)
    d.update(kw)
    return L.VsgDebugConvF32(**d)


@pytest.mark.parametrize("bad", [
    dict(x=None), dict(w=None), dict(y=None), dict(B=0), dict(Cin=0), dict(Lin=0), dict(Cout=0), dict(k=0), dict(dil=0),
    dict(Lq=0), dict(out_stride=0), dict(out_phase=1), dict(Lq=65), dict(Lout=63, Lq=64), dict(epi=5), dict(epi=-1),
    dict(epi=1, Cout=3), dict(epi=4, Cout=1), dict(gate_interleave=1), dict(x_cs=63), dict(x_bs=63),
    dict(mask=1, mask_bs=63), dict(bcond=1, bcond_bs=0), dict(acc_mode=3), dict(acc_mode=1, epi=3),
    dict(acc_mode=2, acc_div=0.0), dict(res=1, epi=2), dict(res=1, res_cs=63, res_bs=64), dict(epi=3, couple_sign=0),
    dict(epi=2, rs_split=2), dict(epi=2, rs_split=-1), dict(epi=2, rs_split=0, y2=None), dict(y_cs=63),
    dict(Cout=2, y_bs=64),
])
def test_conv_f32_hook_rejects_bad_arguments_without_a_device(bad):
    L = _lib()
    d = _desc(**bad)
    assert L.lib().vsg_debug_conv_f32(ctypes.byref(d), None, 0) == -1, bad
    assert L.lib().vsg_debug_conv_f32(None, None, 0) == -1


def test_other_f32_hooks_reject_bad_arguments_without_a_device():
    lib = _lib().lib()
    up = lib.vsg_debug_upsample_f32
    ok = dict(x=1, w=1, bias=1, Cin=4, Cout=2, rate=2, k=4, B=1, Lin=8, y=1)
    for bad in (dict(x=None), dict(w=None), dict(bias=None), dict(y=None), dict(Cin=0), dict(Cout=0), dict(rate=0),
                dict(k=1), dict(k=5), dict(B=0), dict(Lin=0)):
        a = dict(ok, **bad)
        assert up(a["x"], a["w"], a["bias"], a["Cin"], a["Cout"], a["rate"], a["k"], a["B"], a["Lin"], a["y"], 0) == -1, bad
    post = lib.vsg_debug_conv_post_f32
    ok = dict(x=1, w=1, C=16, L=100, k=7, slope=0.1, B=1, n0=0, n1=100, wav=1, ld=100)
    for bad in (dict(x=None), dict(w=None), dict(wav=None), dict(C=0), dict(L=0), dict(k=0), dict(B=0), dict(n0=-1),
                dict(n1=0), dict(n0=50, n1=50), dict(n1=101), dict(ld=99)):
        a = dict(ok, **bad)
        assert post(a["x"], a["w"], a["C"], a["L"], a["k"], a["slope"], a["B"], a["n0"], a["n1"], a["wav"], a["ld"], 0) == -1, bad
    cond = lib.vsg_debug_cond_f32
    ok = dict(W=1, bias=None, g=1, out=1, O=4, I=4, B=1)
    for bad in (dict(W=None), dict(g=None), dict(out=None), dict(O=0), dict(I=0), dict(B=0)):
        a = dict(ok, **bad)
        assert cond(a["W"], a["bias"], a["g"], a["out"], a["O"], a["I"], a["B"], 0) == -1, bad
