"""Times the whole model four ways, in one process, variants alternated after warm-up (full hparams, seeded weights):

  forward   VISinger.forward(infer=True): the prior network's PyTorch glue between ~10 library calls;
  graphed   VISinger.forward_graphed: the same captured into one PyTorch-side CUDA graph per shape;
  native    VISinger.forward_native: one vsg_model_forward call (eager);
  c-graph   vsg_model_forward captured in a torch.cuda.CUDAGraph (what a C caller can capture itself).

Configs: B = 1 x T = 400 (BASELINE config 1) and B = 16 x T = 1000, each in bf16 and bf16x3.  Per call: device time from
CUDA events around `--reps` back-to-back calls; for the eager variants also the host time of the enqueue (host clock
around the calls, before the synchronise).  L2 is not flushed (back-to-back inference).  Prints the card's name, power
limit and maximum SM clock first.

    python tools/time_native_model.py [--reps 20] [--rounds 3]"""
import argparse
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from model_inputs import full_model_mirror, synth_utterances  # noqa: E402
from visinger_b200 import _lib  # noqa: E402


def measure(fn, reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    h0 = time.perf_counter()
    for _ in range(reps):
        fn()
    h1 = time.perf_counter()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, (h1 - h0) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_native_model.py needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print(f"card: {q.stdout.strip() or q.stderr.strip()}", flush=True)
    dev = torch.device("cuda:0")
    for prec in ("bf16", "bf16x3"):
        m = full_model_mirror(precision=prec).to(dev)
        for B, T in ((1, 400), (16, 1000)):
            b = synth_utterances(seed=B * T, n=B, lengths=[T] * B)
            args = [b[k].to(dev) for k in ("text_tokens", "note_pitch", "note_dur", "mel2ph")]
            spk = b["spk_ids"].to(dev)
            noise = torch.randn(B, 192, T, generator=torch.Generator().manual_seed(1)).to(dev)
            T_ph = args[0].shape[1]
            # the C caller's view: fixed buffers, host speaker ids, one captured call
            pack = m._model_pack(dev)
            code = _lib.precision_code(prec)
            ws = torch.empty(pack.workspace_bytes(B, T_ph, T, code), dtype=torch.uint8, device=dev)
            wav = torch.empty(B, T * pack.hop, device=dev)
            spk_h = b["spk_ids"].contiguous()
            L = _lib.lib()

            def c_call():
                rc = L.vsg_model_forward(pack.handle, *[t.data_ptr() for t in args], spk_h.data_ptr(), None, None, None,
                                         noise.data_ptr(), None, wav.data_ptr(), None, None, B, T_ph, T, code,
                                         ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
                _lib.check(rc, "vsg_model_forward")

            c_call()
            launches = L.vsg_last_launch_count()
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                with torch.cuda.graph(g, stream=side):
                    c_call()
            torch.cuda.synchronize()
            variants = {
                "forward": lambda: m(*args, spk_id=spk, infer=True, noise=noise),
                "graphed": lambda: m.forward_graphed(*args, spk_id=spk, noise=noise),
                "native": lambda: m.forward_native(*args, spk_id=spk_h, noise=noise),   # host ids: no device sync
                "c-graph": g.replay,
            }
            for fn in variants.values():      # warm-up: packs, workspaces, graph captures
                fn()
                fn()
            ref = m(*args, spk_id=spk, infer=True, noise=noise)["wav_out"]
            nat = m.forward_native(*args, spk_id=spk_h, noise=noise)["wav_out"]
            g.replay()
            torch.cuda.synchronize()
            rel = float((nat - ref).norm() / ref.norm())
            res = {k: [] for k in variants}
            for _ in range(a.rounds):
                for k, fn in variants.items():
                    res[k].append(measure(fn, a.reps))
            line = ", ".join(f"{k} {min(d for d, _ in v):.3f} ms" + (f" (host {min(h for _, h in v):.3f} ms)"
                                                                      if k in ("forward", "native") else "")
                             for k, v in res.items())
            print(f"{prec} B={B} T={T} (T_ph={T_ph}, {launches} launches in vsg_model_forward): {line}; "
                  f"native vs forward rel-L2 {rel:.2e}, c-graph == native: {torch.equal(wav, nat)}", flush=True)


if __name__ == "__main__":
    main()
