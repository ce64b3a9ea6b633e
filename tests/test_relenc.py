"""RelativeEncoder (modules/rel_transformer.py:257-320; SURVEY.md section 8 row f1).

CPU: the oracle (its own formulation of the banded relative-position terms) against fixtures generated from the UNMODIFIED
reference module (tests/golden/make_golden_relenc.py).  GPU: `vsg_relenc_forward` through the module mirror against the
same fixtures, fp32 mode, at 2e-5 (the fp32-vs-fp64 floor of the reference itself is 1.5e-6 on these cases)."""
import pytest
import torch

from oracle import visinger_oracle as O
from helpers import load_npz, weights_of, maxabs

SMALL = ["small_relenc", "small_relenc_gframe", "small_relenc_nog"]


def _cfg(z):
    return {str(k): int(v) for k, v in zip(z["cfg_keys"], z["cfg_vals"])}


def _okw(cfg):
    return dict(n_heads=cfg["n_heads"], n_layers=cfg["n_layers"], kernel_size=cfg["kernel_size"], window=cfg["window"])


def _full_case():
    z = load_npz("full_relenc")
    cfg = _cfg(z)
    seed, B, T = int(z["seed"]), int(z["B"]), int(z["T"])
    sd = O.synth_rel_encoder_state_dict(O.rel_encoder_param_shapes(cfg["hidden"], cfg["filter"], cfg["n_heads"], cfg["n_layers"],
                                                                   cfg["kernel_size"], cfg["window"], cfg["gin"] or None), seed)
    gen = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, cfg["hidden"], T, generator=gen)
    g = torch.randn(B, cfg["gin"], T if int(z["g_t"]) else 1, generator=gen)
    mask = torch.ones(B, 1, T)
    for b, n in enumerate(z["lengths"].tolist()):
        mask[b, :, n:] = 0
    return z, cfg, sd, x, mask, g


@pytest.mark.parametrize("name", SMALL)
def test_oracle_small_golden(name):
    z = load_npz(name)
    cfg, sd = _cfg(z), weights_of(z)
    x, mask = torch.from_numpy(z["x"]), torch.from_numpy(z["mask"])
    g = torch.from_numpy(z["g"]) if cfg["gin"] else None
    with torch.no_grad():
        y = O.rel_encoder(sd, x, mask, g, **_okw(cfg))
    assert maxabs(y, torch.from_numpy(z["y"])) <= 2e-6
    assert float((y * (1 - mask)).abs().max()) == 0.0 and float(y.abs().max()) > 1.0


def test_oracle_full_config_golden():
    z, cfg, sd, x, mask, g = _full_case()
    with torch.no_grad():
        y = O.rel_encoder(sd, x, mask, g, **_okw(cfg))
    assert maxabs(y[:, ::7, ::int(z["slice_t"])], torch.from_numpy(z["y"])) <= 1e-5


def test_torch_statement_matches_the_oracle():
    """The module's PyTorch statement (diagonal views) and the oracle (gather / scatter) are two formulations of
    rel_transformer.py:137-177; both must agree with the reference fixture."""
    from visinger_b200.modules.rel_transformer import RelativeEncoder
    z = load_npz("small_relenc")
    cfg, sd = _cfg(z), weights_of(z)
    m = RelativeEncoder(cfg["hidden"], cfg["filter"], cfg["n_heads"], cfg["n_layers"], kernel_size=cfg["kernel_size"],
                        window_size=cfg["window"], gin_channels=cfg["gin"]).eval()
    m.load_state_dict(sd, strict=True)
    with torch.no_grad():
        y = m(torch.from_numpy(z["x"]), torch.from_numpy(z["mask"]), torch.from_numpy(z["g"]))
    assert maxabs(y, torch.from_numpy(z["y"])) <= 2e-5


def _build(cfg, sd, device):
    from visinger_b200.modules.rel_transformer import RelativeEncoder
    m = RelativeEncoder(cfg["hidden"], cfg["filter"], cfg["n_heads"], cfg["n_layers"], kernel_size=cfg["kernel_size"],
                        window_size=cfg["window"], gin_channels=cfg["gin"] or None)
    m.load_state_dict(sd, strict=True)
    return m.to(device).eval()


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
def test_relenc_fp32_small_golden(cuda_device, name):
    z = load_npz(name)
    cfg, sd = _cfg(z), weights_of(z)
    m = _build(cfg, sd, cuda_device)
    x, mask = torch.from_numpy(z["x"]).to(cuda_device), torch.from_numpy(z["mask"]).to(cuda_device)
    g = torch.from_numpy(z["g"]).to(cuda_device) if cfg["gin"] else None
    y = m(x, mask, g)
    err = maxabs(y.cpu(), torch.from_numpy(z["y"]))
    print(f"relenc fp32 {name}: max-abs {err:.3e}")
    assert err <= 2e-5
    assert float((y * (1 - mask)).abs().max()) == 0.0
    assert torch.equal(y, m(x, mask, g))
    # the library really ran (no PyTorch fallback): its launch counter moved
    import visinger_b200
    assert visinger_b200.last_launch_count() >= 7 * cfg["n_layers"]


@pytest.mark.gpu
def test_relenc_fp32_full_config_golden(cuda_device):
    z, cfg, sd, x, mask, g = _full_case()
    m = _build(cfg, sd, cuda_device)
    y = m(x.to(cuda_device), mask.to(cuda_device), g.to(cuda_device))
    err = maxabs(y.cpu()[:, ::7, ::int(z["slice_t"])], torch.from_numpy(z["y"]))
    with torch.no_grad():
        yo = O.rel_encoder(sd, x, mask, g, **_okw(cfg))
    err_o = maxabs(y.cpu(), yo)
    print(f"relenc fp32 full: max-abs vs reference fixture {err:.3e}, vs oracle (all elements) {err_o:.3e}")
    assert err <= 2e-5 and err_o <= 2e-5


@pytest.mark.gpu
def test_relenc_long_sequence_vs_oracle(cuda_device):
    """T = 1000 (bench length; 16 key tiles, ragged last tile), per-utterance condition like the PitchPredictor."""
    cfg = dict(hidden=192, filter=768, n_heads=2, n_layers=2, kernel_size=9, window=4, gin=16)
    sd = O.synth_rel_encoder_state_dict(O.rel_encoder_param_shapes(192, 768, 2, 2, 9, 4, 16), 31)
    gen = torch.Generator().manual_seed(32)
    x, g = torch.randn(2, 192, 1000, generator=gen), torch.randn(2, 16, 1, generator=gen)
    mask = torch.ones(2, 1, 1000)
    mask[1, :, 777:] = 0
    with torch.no_grad():
        yo = O.rel_encoder(sd, x, mask, g, **_okw(cfg))
    m = _build(cfg, sd, cuda_device)
    y = m(x.to(cuda_device), mask.to(cuda_device), g.to(cuda_device))
    err = maxabs(y.cpu(), yo)
    print(f"relenc fp32 T=1000: max-abs {err:.3e}")
    assert err <= 2e-5


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
def test_relenc_bf16_small_vs_reference(cuda_device, name):
    """Throughput mode: tcgen05 projections / FFN, warp-mma flash attention, bf16 activations."""
    z = load_npz(name)
    cfg, sd = _cfg(z), weights_of(z)
    m = _build(cfg, sd, cuda_device)
    m.precision = "bf16"
    x, mask = torch.from_numpy(z["x"]).to(cuda_device), torch.from_numpy(z["mask"]).to(cuda_device)
    g = torch.from_numpy(z["g"]).to(cuda_device) if cfg["gin"] else None
    y = m(x, mask, g)
    ref = torch.from_numpy(z["y"])
    rel = float((y.cpu() - ref).norm() / ref.norm())
    print(f"relenc bf16 {name}: rel-L2 {rel:.3e} max-abs {maxabs(y.cpu(), ref):.3e}")
    assert rel <= 8e-3 and maxabs(y.cpu(), ref) <= 0.06          # 1.5x the measured 5.0e-3 / 4.0e-2
    assert float((y * (1 - mask)).abs().max()) == 0.0
    assert torch.equal(y, m(x, mask, g))


@pytest.mark.gpu
def test_relenc_bf16_full_config_vs_oracle(cuda_device):
    z, cfg, sd, x, mask, g = _full_case()
    with torch.no_grad():
        yo = O.rel_encoder(sd, x, mask, g, **_okw(cfg))
    m = _build(cfg, sd, cuda_device)
    m.precision = "bf16"
    y = m(x.to(cuda_device), mask.to(cuda_device), g.to(cuda_device))
    rel = float((y.cpu() - yo).norm() / yo.norm())
    print(f"relenc bf16 full: rel-L2 {rel:.3e} max-abs {maxabs(y.cpu(), yo):.3e}")
    assert rel <= 8.5e-3 and maxabs(y.cpu(), yo) <= 0.09       # 1.5x the measured 5.6e-3 / 5.8e-2


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,n_heads", [(64, 2), (128, 2)])
@pytest.mark.parametrize("window", [1, 7])
@pytest.mark.parametrize("T", [129, 1000, 2048])
def test_relenc_bf16_head_widths_and_windows_vs_oracle(cuda_device, hidden, n_heads, window, T):
    """bf16 encoder at head widths 32 and 64, windows 1 and 7, up to the 16 key tiles of T = 2048, one ragged utterance;
    the full-config gates (measured at most 4.6e-3 / 4.7e-2 on a B200)."""
    cfg = dict(hidden=hidden, filter=4 * hidden, n_heads=n_heads, n_layers=2, kernel_size=9, window=window, gin=16)
    sd = O.synth_rel_encoder_state_dict(O.rel_encoder_param_shapes(hidden, 4 * hidden, n_heads, 2, 9, window, 16), hidden + window)
    gen = torch.Generator().manual_seed(T + window)
    x, g = torch.randn(2, hidden, T, generator=gen), torch.randn(2, 16, 1, generator=gen)
    mask = torch.ones(2, 1, T)
    mask[1, :, T * 2 // 3:] = 0
    with torch.no_grad():
        yo = O.rel_encoder(sd, x, mask, g, **_okw(cfg))
    m = _build(cfg, sd, cuda_device)
    m.precision = "bf16"
    y = m(x.to(cuda_device), mask.to(cuda_device), g.to(cuda_device)).cpu()
    rel = float((y - yo).norm() / yo.norm())
    print(f"relenc bf16 hidden={hidden} heads={n_heads} w={window} T={T}: rel-L2 {rel:.3e} max-abs {maxabs(y, yo):.3e}")
    assert rel <= 8.5e-3 and maxabs(y, yo) <= 0.09
    assert float((y * (1 - mask)).abs().max()) == 0.0
