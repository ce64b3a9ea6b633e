"""Shared builders for the parity tests: golden-fixture loading and seeded cases."""
import ast
import os

import numpy as np
import torch

from oracle import visinger_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

from visinger_b200.configs import VISINGER_FLOW as FLOW_FULL, VISINGER_GENERATOR as GEN_FULL  # noqa: E402


def load_npz(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)


PART_BYTES = 800_000        # array bytes per fixture file: random float32 weights barely compress, and files stay < 1 MB


def _part_path(name, i):
    return os.path.join(GOLDEN, name + (f"_part{i}" if i else "") + ".npz")


def save_npz_parts(name, arrays):
    """np.savez_compressed of `arrays` into GOLDEN/<name>.npz, continued in <name>_part1.npz, <name>_part2.npz, ...
    whenever a file would hold more than PART_BYTES of array data."""
    parts, size = [{}], 0
    for k, v in arrays.items():
        if parts[-1] and size + v.nbytes > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += v.nbytes
    for i, p in enumerate(parts):
        np.savez_compressed(_part_path(name, i), **p)
    i = len(parts)
    while os.path.exists(_part_path(name, i)):          # parts left over from a larger earlier fixture
        os.remove(_part_path(name, i))
        i += 1


def load_npz_parts(name):
    """The arrays of <name>.npz and of its continuation files (save_npz_parts) as one dict."""
    out, i = {}, 0
    while os.path.exists(_part_path(name, i)):
        with np.load(_part_path(name, i), allow_pickle=False) as z:
            out.update({k: z[k] for k in z.files})
        i += 1
    return out


def flow_cfg_of(z):
    return {k: int(v) for k, v in zip(z["cfg_keys"].tolist(), z["cfg_vals"].tolist())}


def gen_cfg_of(z):
    return ast.literal_eval(str(z["cfg_json"]))


def weights_of(z):
    return {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w/")}


def flow_oracle_kw(cfg):
    return dict(channels=cfg["channels"], hidden=cfg["hidden"], kernel_size=cfg["kernel_size"],
                dilation_rate=cfg["dilation_rate"], n_layers=cfg["n_layers"], n_flows=cfg["n_flows"])


def gen_oracle_kw(cfg):
    return dict(resblock=cfg["resblock"], resblock_kernel_sizes=cfg["rk"], resblock_dilation_sizes=cfg["rd"],
                upsample_rates=cfg["ur"], upsample_kernel_sizes=cfg["uk"])


def flow_shapes(cfg):
    return O.flow_param_shapes(cfg["channels"], cfg["hidden"], cfg["kernel_size"], cfg["n_layers"], cfg["n_flows"],
                               cfg["gin"])


def gen_shapes(cfg):
    return O.generator_param_shapes(cfg["initial_channel"], cfg["resblock"], cfg["rk"], cfg["rd"], cfg["ur"],
                                    cfg["uic"], cfg["uk"], cfg["gin"])


def make_inputs(seed, B, C, T, gin, lengths=None):
    """Same recipe as tests/golden/make_golden.py::_inputs."""
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, T, generator=gen)
    g = 0.1 * torch.randn(B, gin, 1, generator=gen) if gin else None
    mask = torch.ones(B, 1, T)
    if lengths is not None:
        for b, n in enumerate(lengths):
            mask[b, :, n:] = 0
    return x, mask, g


def build_flow(cfg, sd, device, precision="fp32"):
    from visinger_b200 import ResidualCouplingBlock
    m = ResidualCouplingBlock(cfg["channels"], cfg["hidden"], cfg["kernel_size"], cfg["dilation_rate"],
                              cfg["n_layers"], n_flows=cfg["n_flows"], gin_channels=cfg["gin"], precision=precision)
    m.load_state_dict(sd)
    return m.to(device).eval()


def build_gen(cfg, sd, device, precision="fp32"):
    from visinger_b200 import Generator
    m = Generator(cfg["initial_channel"], cfg["resblock"], cfg["rk"], cfg["rd"], cfg["ur"], cfg["uic"], cfg["uk"],
                  gin_channels=cfg["gin"], precision=precision)
    m.load_state_dict(sd)
    return m.to(device).eval()


def maxabs(a, b):
    return float((a.double() - b.double()).abs().max()) if a.numel() else 0.0
