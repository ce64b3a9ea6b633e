"""The fp32 FFMA kernels (csrc/kernels_f32.cuh) one launch at a time, through vsg_debug_conv_f32, vsg_debug_upsample_f32,
vsg_debug_conv_post_f32 and vsg_debug_cond_f32, against the float64 statements of tests/conv_f32_reference.py on both
operand layers: exact operands (every sum exact in fp32: equal values, or the ulp bounds of tanhf / expf / sqrtf) and
random operands (the provable fp32 FMA bound gamma_{n+m} * S).

Every convolution case runs B = 3 different utterances with NaN in every element the kernel must not read (the input
rows past Lin, a guard channel past Cin, the mask past Lout, bcond past Cout, res past Lout and past Cout) and outputs
pre-filled with a sentinel, with guard elements past each row and a guard channel past the last one; elements the launch
does not write must keep their bits.  A second call must give the same bits, and each utterance must equal its B = 1
run (the same buffers, offset to that utterance) bit for bit.

Floors, the worst |got - float64| / S over the random operands of this module, measured on an NVIDIA B200 at a 1000 W
power limit (the gates are the derived bounds, not these numbers; MAG's S includes the magnitude itself):
  conv linear 4.4e-7, gate 9.0e-8, res_skip 3.3e-7, couple 2.3e-7, mag 1.1e-7; upsample 4.3e-7; conv_post 1.7e-7;
  cond GEMV 1.1e-7.
"""
import pytest
import torch

import conv_f32_reference as R

pytestmark = pytest.mark.gpu

SENTINEL = 12345.0
NAN = float("nan")
_floors = {}


def _note(name, value):
    _floors[name] = max(_floors.get(name, 0.0), value)
    print(f"floor[{name}] so far {_floors[name]:.3e}")


def _lib():
    from visinger_b200 import _lib
    return _lib


def _reads_y(c):
    return (c["epi"] == R.LINEAR and (c["acc_mode"] != R.ACC_SET or c["res"] == "alias")) or c["epi"] == R.RES_SKIP or \
        (c["epi"] == R.COUPLE and c["res"] != "sep")


def _buffers(c, op, dev):
    """The launch's device buffers (padded, guarded) and the initial content of its outputs."""
    B, Cin, Lin, Cout, Lout = c["B"], c["Cin"], c["Lin"], c["Cout"], c["Lout"]
    ych = R.ychannels(c)
    ny2 = Cout - c["rs_split"] if c["epi"] == R.RES_SKIP else 0
    x = torch.full((B, Cin + 1, Lin + 3), NAN)
    x[:, :Cin, :Lin] = op["x"]
    bufs = dict(x=x)
    if op["mask"] is not None:
        bufs["mask"] = R.mask_buffer(c, op["mask"]).reshape(B, Lout + 5)
    if op["bcond"] is not None:
        bc = torch.full((B, Cout + 3), NAN)
        bc[:, :Cout] = op["bcond"]
        bufs["bcond"] = bc
    if c["res"] == "sep":
        r = torch.full((B, Cout + 1, Lout + 2), NAN)
        r[:, :Cout, :Lout] = op["res"]
        bufs["res"] = r
    if ych:
        y = torch.full((B, ych + 1, Lout + 3), SENTINEL)
        if _reads_y(c):
            y[:, :ych, :Lout] = op["y_old"]
        bufs["y"] = y
    if ny2:
        y2 = torch.full((B, ny2 + 1, Lout + 3), SENTINEL)
        y2[:, :ny2, :Lout] = NAN if c["y2_first"] else op["y2_old"]
        bufs["y2"] = y2
    return {k: v.to(dev).contiguous() for k, v in bufs.items()}


def _launch(c, op, bufs, B=None, b0=0):
    """One hook call on utterances [b0, b0 + B) of the buffers (B = 1: a single utterance at its offset)."""
    B = c["B"] if B is None else B
    sl = {k: v[b0:b0 + B] for k, v in bufs.items()}
    Lout, Cout = c["Lout"], c["Cout"]
    kw = dict(B=B, Cin=c["Cin"], Lin=c["Lin"], Lq=c["Lq"], Lout=Lout, x_cs=c["Lin"] + 3,
              x_bs=(c["Cin"] + 1) * (c["Lin"] + 3), dil=c["dil"], in_off0=c["in_off0"], pre_lrelu=c["pre_lrelu"],
              slope=op["slope"], out_stride=c["out_stride"], out_phase=c["out_phase"], epi=c["epi"],
              acc_mode=c["acc_mode"], acc_div=float(c["nk"]), rs_split=c["rs_split"], y2_first=c["y2_first"],
              y2_mask=c["y2_mask"], couple_sign=c["couple_sign"], gate_interleave=c["gate_interleave"])
    if "y" in sl:
        kw.update(y=sl["y"], y_cs=Lout + 3, y_bs=sl["y"].shape[1] * (Lout + 3))
    if "y2" in sl:
        kw.update(y2=sl["y2"], y2_cs=Lout + 3, y2_bs=sl["y2"].shape[1] * (Lout + 3))
    if "mask" in sl:
        kw.update(mask=sl["mask"], mask_bs=Lout + 5)
    if "bcond" in sl:
        kw.update(bcond=sl["bcond"], bcond_bs=Cout + 3)
    if c["res"] == "sep":
        kw.update(res=sl["res"], res_cs=Lout + 2, res_bs=(Cout + 1) * (Lout + 2))
    elif c["res"] == "alias":
        kw.update(res=sl["y"], res_cs=Lout + 3, res_bs=kw["y_bs"])
    return _lib().debug_conv_f32(sl["x"], op["w"], op["bias"], **kw)


def _run_case(c, layer, dev):
    op = R.operands(c, layer)
    bufs = _buffers(c, op, dev)
    init = {k: v.cpu().clone() for k, v in bufs.items()}
    tile, _ = _launch(c, op, bufs)
    plan = _lib().debug_conv_f32_plan(c["Cout"], c["k"], c["dil"])
    assert tile == plan[:2], (tile, plan)
    got = {k: bufs[k].cpu() for k in ("y", "y2") if k in bufs}
    for name, (V, T, Wr, S) in R.conv_ref(c, op, layer).items():
        Lout, ch = c["Lout"], V.shape[1]
        g, i0 = got[name], init[name]
        ok, ratio = R.compare(g[:, :ch, :Lout], i0[:, :ch, :Lout], V, T, Wr)
        assert ok, (c["name"], layer, name, ratio)
        # guards: the channel past the last and the row tails keep their initial bits
        guard = torch.ones_like(g, dtype=torch.bool)
        guard[:, :ch, :Lout] = False
        assert torch.equal(g[guard].view(torch.int32), i0[guard].view(torch.int32)), (c["name"], name, "guard")
        if layer == "random" and bool(Wr.any()):
            d = (g[:, :ch, :Lout].double() - V).abs()[Wr]
            _note(f"conv {['linear', 'gate', 'res_skip', 'couple', 'mag'][c['epi']]}", float((d / S[Wr].clamp_min(R.TINY)).max()))
    # a second call gives the same bits
    again = _buffers(c, op, dev)
    _launch(c, op, again)
    for k in got:
        assert torch.equal(again[k].cpu().view(torch.int32), got[k].view(torch.int32)), (c["name"], "repeat")
    # each utterance alone, read and written at its own offset, gives the bits of the batched launch
    for b in range(c["B"]):
        solo = _buffers(c, op, dev)
        _launch(c, op, solo, B=1, b0=b)
        for k in got:
            assert torch.equal(solo[k][b].cpu().view(torch.int32), got[k][b].view(torch.int32)), (c["name"], "B=1", b)


CASES = R.gpu_cases()


@pytest.mark.parametrize("layer", ["exact", "random"])
@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_conv_f32_launch(c, layer, cuda_device):
    _run_case(c, layer, cuda_device)


def test_conv_f32_refuses_a_window_over_200kb_without_a_launch(cuda_device):
    c = R.SMEM_REFUSED
    op = R.operands(c, "exact")
    bufs = _buffers(c, op, cuda_device)
    before = bufs["y"].cpu().clone()
    _, rc = _lib().debug_conv_f32(bufs["x"], op["w"], op["bias"], B=c["B"], Cin=c["Cin"], Lin=c["Lin"], Lq=c["Lq"],
                                     x_cs=c["Lin"] + 3, x_bs=(c["Cin"] + 1) * (c["Lin"] + 3), dil=c["dil"],
                                     in_off0=c["in_off0"], y=bufs["y"], y_cs=c["Lout"] + 3,
                                     y_bs=(c["Cout"] + 1) * (c["Lout"] + 3), check_rc=False)
    assert rc == -4 and _lib().last_launch_count() == 0
    assert torch.equal(bufs["y"].cpu().view(torch.int32), before.view(torch.int32))


@pytest.mark.parametrize("layer", ["exact", "random"])
@pytest.mark.parametrize("shape", R.UPS_SHAPES, ids=[f"{a}x{b}-r{r}-k{k}" for a, b, r, k in R.UPS_SHAPES])
def test_upsample_f32(shape, layer, cuda_device):
    Cin, Cout, rate, k = shape
    for Lin in R.UPS_LINS:
        x, w, b = R.ups_operands(Cin, Cout, rate, k, 3, Lin, layer, 100 * rate + k + Lin)
        want, tol, S = R.upsample_ref(x, w, b, rate, layer)
        xd = x.to(cuda_device).contiguous()
        ys = []
        for _ in range(2):
            y = torch.full((3, Cout, Lin * rate), SENTINEL, device=cuda_device)
            _lib().debug_upsample_f32(xd, w, b, rate, y)
            assert _lib().last_launch_count() == rate
            ys.append(y.cpu())
        y = ys[0]
        assert torch.equal(ys[1].view(torch.int32), y.view(torch.int32))
        ok, ratio = R.compare(y, torch.full_like(y, SENTINEL), want, tol, torch.ones_like(y, dtype=torch.bool))
        assert ok, (shape, Lin, layer, ratio)
        if layer == "random":
            _note("upsample", float(((y.double() - want).abs() / S.clamp_min(R.TINY)).max()))
        for bb in range(3):
            solo = torch.full((1, Cout, Lin * rate), SENTINEL, device=cuda_device)
            _lib().debug_upsample_f32(xd[bb:bb + 1], w, b, rate, solo)
            assert torch.equal(solo[0].cpu().view(torch.int32), y[bb].view(torch.int32))


@pytest.mark.parametrize("layer", ["exact", "random"])
@pytest.mark.parametrize("post", R.POST_CASES, ids=[f"C{a}-k{b}-L{c}" for a, b, c in R.POST_CASES])
def test_conv_post_f32(post, layer, cuda_device):
    C, k, L = post
    x, w, slope = R.post_operands(C, k, L, 3, layer, C + 10 * k + L)
    xd = x.to(cuda_device).contiguous()
    for n0, n1 in ((0, L), (37, L - 200), (L - 1, L)):
        ld = n1 - n0 + 5
        want, tol, S = R.post_ref(x, w, slope, n0, n1, layer)
        outs = []
        for _ in range(2):
            wav = torch.full((3 * ld + 4,), SENTINEL, device=cuda_device)
            _lib().debug_conv_post_f32(xd, w, slope, n0, n1, wav, ld)
            outs.append(wav.cpu())
        wav = outs[0]
        assert torch.equal(outs[1].view(torch.int32), wav.view(torch.int32))
        rows = torch.stack([wav[b * ld:b * ld + n1 - n0] for b in range(3)])
        ok, ratio = R.compare(rows, torch.full_like(rows, SENTINEL), want, tol, torch.ones_like(rows, dtype=torch.bool))
        assert ok, (post, n0, n1, layer, ratio)
        tail = torch.cat([wav[b * ld + n1 - n0:(b + 1) * ld] for b in range(3)] + [wav[3 * ld:]])
        assert bool((tail == SENTINEL).all()), "conv_post wrote past n1 - n0"
        if layer == "random":
            _note("conv_post", float(((rows.double() - want).abs() / S.clamp_min(R.TINY)).max()))


@pytest.mark.parametrize("layer", ["exact", "random"])
@pytest.mark.parametrize("cond", R.COND_CASES, ids=[f"O{a}-I{b}-B{c}" for a, b, c in R.COND_CASES])
def test_cond_gemv_f32(cond, layer, cuda_device):
    O, I, B = cond
    W, bias, g = R.cond_operands(O, I, B, layer, O + I + B)
    want, tol, S = R.cond_ref(W, bias, g, layer)
    dev = cuda_device
    Wd, bd, gd = (t.to(dev).contiguous() for t in (W, bias, g))
    out = torch.full((B * O + 7,), SENTINEL, device=dev)
    _lib().debug_cond_f32(Wd, bd, gd, out)
    got = out.cpu()
    assert bool((got[B * O:] == SENTINEL).all())
    got = got[:B * O].reshape(B, O)
    ok, ratio = R.compare(got, torch.full_like(got, SENTINEL), want, tol, torch.ones_like(got, dtype=torch.bool))
    assert ok, (cond, layer, ratio)
    if layer == "random":
        _note("cond", float(((got.double() - want).abs() / S.clamp_min(R.TINY)).max()))
    out2 = torch.full((B * O + 7,), SENTINEL, device=dev)
    _lib().debug_cond_f32(Wd, bd, gd, out2)
    assert torch.equal(out2.cpu()[:B * O].reshape(B, O).view(torch.int32), got.view(torch.int32))
    out0 = torch.full((B * O,), SENTINEL, device=dev)
    _lib().debug_cond_f32(Wd, None, gd, out0)
    want0, tol0, _ = R.cond_ref(W, None, g, layer)
    g0 = out0.cpu().reshape(B, O)
    assert R.compare(g0, torch.full_like(g0, SENTINEL), want0, tol0, torch.ones_like(g0, dtype=torch.bool))[0]


def test_print_floors():
    """(Runs last in the module) the worst |err| / S per kernel over the random operands."""
    for k, v in sorted(_floors.items()):
        print(f"FLOOR {k}: {v:.3e}")
