"""Times voice conversion (vsg_model_convert) on the GPU, full hparams with seeded weights (win_length 1200):

  spectrogram   vsg_spectrogram alone at B = 16 x T = 1000: tcgen05 (bf16) against the FFMA kernel (fp32);
  chain         the existing public calls one after another: vsg_spectrogram -> vsg_posterior_forward ->
                vsg_flow_forward(reverse=0) -> vsg_infer_zp (speaker conditions gathered by the caller beforehand);
  native        one vsg_model_convert call from the waveform (eager);
  c-graph       the same call captured in a torch.cuda.CUDAGraph.

Configs: B = 1 x T = 400 and B = 16 x T = 1000, each in bf16 and bf16x3.  Device time from CUDA events around `--reps`
back-to-back calls, variants alternated over `--rounds`; the best round is printed.  L2 is not flushed.  Prints the card's
name, power limit and maximum SM clock first.

    python tools/time_voice_conversion.py [--reps 20] [--rounds 3]"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from model_inputs import full_hparams  # noqa: E402
from visinger_b200 import _lib  # noqa: E402

PREC = {"fp32": 0, "bf16": 1, "bf16x3": 2}


def measure(fn, reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def model(dev):
    from visinger_b200.models.visinger import VISinger
    hp = full_hparams()
    hp.update(num_spk=4, win_size=1200)
    torch.manual_seed(4321)
    m = VISinger(73, 117, 132, hp).eval()
    with torch.no_grad():
        for f in range(4):
            m.flow.flows[2 * f].post.weight.normal_(0, 0.05)
            m.flow.flows[2 * f].post.bias.normal_(0, 0.05)
    return m.to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_voice_conversion.py needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print(f"card: {q.stdout.strip() or q.stderr.strip()}", flush=True)
    dev = torch.device("cuda:0")
    L = _lib.lib()
    m = model(dev)
    pack = m._convert_pack(dev)
    hop, H = pack.hop, m.hidden_size
    g = torch.Generator().manual_seed(1)

    # the spectrogram alone
    B, T = 16, 1000
    wav = (0.3 * torch.randn(B, T * hop, generator=g)).to(dev)
    ln = torch.full((B,), T, dtype=torch.int32, device=dev)
    spec = torch.empty(B, pack.bins, T, device=dev)
    res = {}
    for r in range(a.rounds):
        for name, prec in (("tcgen05 (bf16)", 1), ("FFMA (fp32)", 0)):
            ws = _lib.workspace(dev, pack.convert_workspace_bytes(B, T, prec))

            def run():
                _lib.check(L.vsg_spectrogram(pack.handle, wav.data_ptr(), ln.data_ptr(), spec.data_ptr(), B, T, prec,
                                             ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)), "vsg_spectrogram")
            run()
            t = measure(run, a.reps)
            res[name] = min(res.get(name, 1e30), t)
    flop = 2.0 * B * T * 2 * pack.bins * 1200
    for name, t in res.items():
        print(f"spectrogram B{B} x T{T} {name}: {t:.3f} ms ({flop / t / 1e9:.1f} TFLOP/s of the DFT-basis GEMM)")

    pe = m.posterior_encoder
    ep = _lib.EncPack(_lib.VsgEncConfig(pe.in_channels, pe.out_channels, pe.hidden_channels, pe.kernel_size,
                                        pe.dilation_rate, pe.n_layers, pe.gin_channels), dict(m.state_dict()),
                      "posterior_encoder.", dev)
    for prec_name in ("bf16", "bf16x3"):
        prec = PREC[prec_name]
        m.precision = m._hot.precision = prec_name
        hot = m._hot._pack()
        for B, T in ((1, 400), (16, 1000)):
            wav = (0.3 * torch.randn(B, T * hop, generator=g)).to(dev)
            ln = torch.full((B,), T, dtype=torch.int32, device=dev)
            mask = torch.ones(B, 1, T, device=dev)
            src = torch.randint(0, 4, (B,), generator=g)
            tgt = torch.randint(0, 4, (B,), generator=g)
            w = m.spk_id_proj.weight.detach()
            g_src, g_tgt = w[src.to(dev)].unsqueeze(-1).contiguous(), w[tgt.to(dev)].unsqueeze(-1).contiguous()
            noise = torch.randn(B, H, T, generator=g).to(dev)
            out = torch.empty(B, T * hop, device=dev)
            z = torch.empty(B, H, T, device=dev)
            z_p = torch.empty(B, H, T, device=dev)
            stats = torch.empty(B, 2 * H, T, device=dev)
            spec = torch.empty(B, pack.bins, T, device=dev)
            ws = torch.empty(pack.convert_workspace_bytes(B, T, prec), dtype=torch.uint8, device=dev)
            ws_e = torch.empty(ep.workspace_bytes(B, T, prec), dtype=torch.uint8, device=dev)
            ws_h = torch.empty(hot.workspace_bytes(B, T, prec), dtype=torch.uint8, device=dev)

            def native():
                _lib.check(L.vsg_model_convert(pack.handle, wav.data_ptr(), None, ln.data_ptr(), src.data_ptr(), None,
                                               tgt.data_ptr(), None, noise.data_ptr(), None, out.data_ptr(), None, None,
                                               B, T, prec, ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)), "vsg_model_convert")

            def chain():
                _lib.check(L.vsg_spectrogram(pack.handle, wav.data_ptr(), ln.data_ptr(), spec.data_ptr(), B, T, prec,
                                             ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)), "vsg_spectrogram")
                _lib.check(L.vsg_posterior_forward(ep.handle, spec.data_ptr(), mask.data_ptr(), g_src.data_ptr(),
                                                   noise.data_ptr(), z.data_ptr(), stats.data_ptr(), B, T, prec,
                                                   ws_e.data_ptr(), ws_e.numel(), _lib.stream_ptr(dev)), "vsg_posterior_forward")
                _lib.check(L.vsg_flow_forward(hot.handle, z.data_ptr(), mask.data_ptr(), g_src.data_ptr(), z_p.data_ptr(),
                                              B, T, 0, prec, ws_h.data_ptr(), ws_h.numel(), _lib.stream_ptr(dev)), "vsg_flow_forward")
                _lib.check(L.vsg_infer_zp(hot.handle, z_p.data_ptr(), mask.data_ptr(), g_tgt.data_ptr(), out.data_ptr(),
                                          None, B, T, prec, ws_h.data_ptr(), ws_h.numel(), _lib.stream_ptr(dev)), "vsg_infer_zp")

            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                native()
                chain()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                native()
            res = {}
            for r in range(a.rounds):
                for name, fn in (("chain", chain), ("native", native), ("c-graph", graph.replay)):
                    fn()
                    res[name] = min(res.get(name, 1e30), measure(fn, a.reps))
            print(f"{prec_name} B{B} x T{T}: " + ", ".join(f"{k} {v:.3f} ms" for k, v in res.items()), flush=True)


if __name__ == "__main__":
    main()
