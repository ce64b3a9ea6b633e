"""Every A/B switch of vsg_set_tc_options (include/visinger_b200.h), turned on alone, on the whole Generator in bf16 and
bf16x3, and the decoder's L2 sub-batching (l2_tensor_mb = 1, min_tiles = 1).

- Each switch must show its effect in the launch count or in the per-image launch counts (vsg_last_launch_images) -- or,
  for a switch that changes the arithmetic of the same launches, in the output bits -- unless it is listed as inert at
  that shape, where it must change neither.  So no case passes vacuously.  Bits 8 (no programmatic dependent launch),
  11 (no N split), 14 (chains on one stream), 26 (row-packed kernel tap by tap), 2 (row-packed kernel as two CTAs per SM)
  and 30 (two epilogue warp sets per block) change launch attributes, tile plans, streams, weight layouts and CTA
  layouts, which the counts do not see: they must leave the counts unchanged.
- Scheduling-only switches (bits 8, 10, 11, 13, 14, 26, 27 and sub-batching) give the default's bits exactly, in both
  modes.  Bit 26 belongs here: the block-Toeplitz form issues the same K = 16 slices per output in the same order as the
  tap-by-tap form (input sub-step, then channel chunk) and only adds slices whose weights are zero, which add exactly 0.
- Switches that change the arithmetic (bits 1, 2, 12, 15, 24, 25, 28-29, 30) are gated against the CPU oracle: bf16
  at the existing gates (full model: rel-L2 5.7e-3, max-abs 5.5e-4, test_gpu_tc.py; ResBlock2 configuration: 1e-2 /
  1.1e-3, test_gpu_round2.py), bf16x3 at 2.5e-6 max-abs.
- The flow's bit 31 (separate res / skip launches) gives the default's bits in bf16 and bf16x3.

bf16x3 floor measured on a B200 (1000 W power limit): waveform max-abs 1.4e-6 against the oracle over every shape and
switch here; gate 2.5e-6.

L2 sub-batching in bf16x3 found a bug: a planar stage output read by a sub-batched next stage at the wrong plane stride
gave max-abs 7.4e-3 at (B, T) = (4, 100) and 4.8e-3 at (2, 171); generator_forward_tc now reads it at B * Lin * Cin.
"""
import pytest
import torch

from oracle import visinger_oracle as O
from helpers import GEN_FULL, FLOW_FULL, build_gen, build_flow, flow_shapes, gen_shapes, make_inputs, maxabs

pytestmark = pytest.mark.gpu

GEN_RB2_TC = dict(initial_channel=32, resblock="2", rk=[3, 5], rd=[[1, 3], [1, 3]], ur=[4, 2], uic=128, uk=[8, 4], gin=16)
CONFIGS = {"full": GEN_FULL, "rb2": GEN_RB2_TC}
SHAPES = [("full", 1, 1), ("full", 3, 17), ("full", 2, 171), ("full", 4, 100), ("rb2", 2, 40)]

DEFAULT = (1, 1, 0, 592)          # halo_mode, w_resident, l2_tensor_mb, min_tiles: the shipped configuration
SCHEDULING = {"bit8": 1 << 8, "bit10": 1 << 10, "bit11": 1 << 11, "bit13": 1 << 13, "bit14": 1 << 14, "bit26": 1 << 26,
              "bit27": 1 << 27, "l2": None}
ARITHMETIC = {"bit1": 1 << 1, "bit2": 1 << 2, "bit12": 1 << 12, "bit15": 1 << 15, "bit24": 1 << 24, "bit25": 1 << 25,
              "bit28": 1 << 28, "bit29": 2 << 28, "bit30": 1 << 30}
# switches whose effect the launch / image counts do not show (see the module docstring)
UNCOUNTED = {"bit8", "bit11", "bit14", "bit26", "bit2", "bit30"}
# bf16 gates of test_gpu_tc.py (full model) and test_gpu_round2.py (ResBlock2 configuration): rel-L2, max-abs
BF16_GATES = {"full": (5.7e-3, 5.5e-4), "rb2": (1.0e-2, 1.1e-3)}
X3_MAXABS = 2.5e-6


def _l2_splits(cfg, B, T):
    """Whether l2_tensor_mb = 1, min_tiles = 1 cuts some stage into sub-batches (plan_sub_batches in csrc/run_tc.cu)."""
    c = CONFIGS[cfg]
    L = T
    for i, rate in enumerate(c["ur"]):
        L *= rate
        per_utt = (c["uic"] >> (i + 1)) * L
        sub = max(1, (1 << 20) // (per_utt * 2))
        if sub * 2 > B:
            sub = B
        if sub < B:
            return True
    return False


def _inert(name, cfg, B, T, prec):
    """(switch, shape, mode) where the switch has nothing to act on under the defaults."""
    full = cfg == "full"
    rp_any = full and T * 300 >= 256          # the row-packed kernel runs the C = 16 stage (T * 300 steps) and up
    if name in UNCOUNTED:
        return True
    if name == "bit1":                        # bf16x3 without the row-packed kernel
        return prec == "bf16" or not rp_any
    if name == "bit24":
        return not rp_any
    if name == "bit25":                       # the row-packed kernel at C = 64 (T * 75 steps; plain bf16 only)
        return prec == "bf16x3" or not full or T * 75 < 256
    if name == "bit15":                       # whole-resblock kernel: plain bf16 ResBlock1, the C = 64 stage
        return prec != "bf16" or not full or T * 75 < 256
    if name == "bit10":                       # bf16x3 merges the upsampler only into planar ResBlock1 stages
        return prec == "bf16x3" and not full
    if name in ("bit28", "bit29"):            # the tcgen05 conv_post needs 16 channels and k = 7 (the full model)
        return not full
    if name == "l2":
        return not _l2_splits(cfg, B, T)
    return False


def _restore():
    from visinger_b200 import _lib
    _lib.set_tc_options(*DEFAULT)


@pytest.fixture(autouse=True)
def _options_restored():
    _restore()
    yield
    _restore()


@pytest.fixture(scope="module")
def oracle_runs():
    """Per (config, B, T): state dict, inputs and the oracle's waveform, computed once."""
    out = {}
    for cfg, B, T in SHAPES:
        c = CONFIGS[cfg]
        sd = O.synth_state_dict(gen_shapes(c), 1234)
        x, _, g = make_inputs(300 + T, B, c["initial_channel"], T, c["gin"])
        kw = dict(resblock=c["resblock"], resblock_kernel_sizes=c["rk"], resblock_dilation_sizes=c["rd"],
                  upsample_rates=c["ur"], upsample_kernel_sizes=c["uk"])
        with torch.no_grad():
            ref = O.generator(sd, x, g, **kw)
        out[(cfg, B, T)] = (sd, x, g, ref)
    return out


_models = {}


def _run(oracle_runs, cfg, B, T, prec, dev):
    from visinger_b200 import _lib
    sd, x, g, _ = oracle_runs[(cfg, B, T)]
    key = (cfg, prec)
    if key not in _models:
        _models[key] = build_gen(CONFIGS[cfg], sd, dev, precision=prec)
    y = _models[key](x.to(dev), g=g.to(dev))
    torch.cuda.synchronize(dev)
    return y.cpu(), _lib.last_launch_count(), _lib.last_launch_images()


def _set(name):
    from visinger_b200 import _lib
    if name == "l2":
        _lib.set_tc_options(1, 1, 1, 1)
    else:
        _lib.set_tc_options((SCHEDULING.get(name) or ARITHMETIC[name]) | 1, 1, 0, 592)


def _check_effect(name, cfg, B, T, prec, base, got, bits_changed=False):
    """A switch shows its effect in the launch / image counts or, for one that changes the arithmetic of the same
    launches, in the output bits; where it has nothing to act on it must change neither."""
    counted = base[1] != got[1] or base[2] != got[2]
    print(f"{name} {cfg} B={B} T={T} {prec}: launches {base[1]} -> {got[1]}, images changed {base[2] != got[2]}, "
          f"bits changed {bits_changed}")
    if name in UNCOUNTED:
        assert not counted, f"{name} changed the launches"
    elif _inert(name, cfg, B, T, prec):
        assert not counted and not bits_changed, f"{name} was expected to be inert here"
    else:
        assert counted or bits_changed, f"{name} changed neither the launches nor the output"


@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
@pytest.mark.parametrize("cfg,B,T", SHAPES)
@pytest.mark.parametrize("name", list(SCHEDULING))
def test_scheduling_switch_keeps_bits(cuda_device, oracle_runs, name, cfg, B, T, prec):
    base = _run(oracle_runs, cfg, B, T, prec, cuda_device)
    _set(name)
    try:
        got = _run(oracle_runs, cfg, B, T, prec, cuda_device)
    finally:
        _restore()
    _check_effect(name, cfg, B, T, prec, base, got)
    assert torch.equal(got[0], base[0]), f"{name}: max-abs {maxabs(got[0], base[0]):.3e} from the default"


@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
@pytest.mark.parametrize("cfg,B,T", SHAPES)
@pytest.mark.parametrize("name", list(ARITHMETIC))
def test_arithmetic_switch_vs_oracle(cuda_device, oracle_runs, name, cfg, B, T, prec):
    ref = oracle_runs[(cfg, B, T)][3]
    base = _run(oracle_runs, cfg, B, T, prec, cuda_device)
    _set(name)
    try:
        got = _run(oracle_runs, cfg, B, T, prec, cuda_device)
    finally:
        _restore()
    y = got[0]
    _check_effect(name, cfg, B, T, prec, base, got, bits_changed=not torch.equal(y, base[0]))
    err = maxabs(y, ref)
    if prec == "bf16":
        rel = float((y - ref).norm() / ref.norm())
        print(f"{name} {cfg} B={B} T={T} bf16: rel-L2 {rel:.3e} max-abs {err:.3e}")
        assert rel <= BF16_GATES[cfg][0] and err <= BF16_GATES[cfg][1]
    else:
        print(f"{name} {cfg} B={B} T={T} bf16x3: max-abs {err:.3e}")
        assert err <= X3_MAXABS


@pytest.mark.parametrize("cfg,B,T", SHAPES)
@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
def test_default_vs_oracle(cuda_device, oracle_runs, cfg, B, T, prec):
    """The reference point of the switch cases: the default configuration against the oracle at the same gates."""
    y = _run(oracle_runs, cfg, B, T, prec, cuda_device)[0]
    ref = oracle_runs[(cfg, B, T)][3]
    if prec == "bf16":
        assert float((y - ref).norm() / ref.norm()) <= BF16_GATES[cfg][0] and maxabs(y, ref) <= BF16_GATES[cfg][1]
    else:
        print(f"default {cfg} B={B} T={T} bf16x3: max-abs {maxabs(y, ref):.3e}")
        assert maxabs(y, ref) <= X3_MAXABS


@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
def test_flow_separate_res_skip_keeps_bits(cuda_device, prec):
    """Bit 31: res and skip as two launches and one cond_layer GEMV per flow, against the merged launches."""
    from visinger_b200 import _lib
    sd = O.synth_state_dict(flow_shapes(FLOW_FULL), 1234)
    flow = build_flow(FLOW_FULL, sd, cuda_device, precision=prec)
    x, mask, g = make_inputs(11, 3, 192, 150, 256, [150, 97, 1])
    args = (x.to(cuda_device) * mask.to(cuda_device), mask.to(cuda_device))
    base = flow(*args, g=g.to(cuda_device), reverse=True).cpu()
    n0 = _lib.last_launch_count()
    _lib.set_tc_options(1 | (1 << 31), 1, 0, 592)
    try:
        got = flow(*args, g=g.to(cuda_device), reverse=True).cpu()
        n1 = _lib.last_launch_count()
    finally:
        _restore()
    assert n1 > n0
    assert torch.equal(got, base)
